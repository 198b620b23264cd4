"""HbvAdj (implicit scheme, csrc/hbv_adj.cu): gradient w.r.t. the forcings and state carry-over
between calls.

  * d loss / d x_phy from the K3 adjoint sweep (lambda^T df/d(P, T, Ep), summed over the nmul
    components) against the float64 oracle (oracle/hbv_adj_oracle.py, whose Newton step gives no
    gradient w.r.t. the forcings: `_NewtonStepForcing` below adds it), per forcing column at the
    parameter-gradient bar RTOL_GRAD, on every adjoint form: the register kernel (shuffle and
    shared-memory nmul reductions), the cp.async-ring kernel (nmul 16, D2) and the no-plane form
    (only x_phy requires grad);
  * the warm-up is differentiable here, so the warm-up rows of x_phy receive gradient too;
  * `cache_states` / `get_states` / `load_states` / `uh_carry_over`: a run stepped chunk by chunk
    equals the one-shot run.
The first test (CPU) pins that forcing gradient to float64 finite differences."""

import contextlib

import pytest
import torch

from conftest import RTOL_FLUX, RTOL_GRAD, STATE_FLOOR, assert_close

gpu = pytest.mark.gpu

D2 = ['parBETA', 'parBETAET']
ALL = ['parBETA', 'parFC', 'parK0', 'parK1', 'parK2', 'parLP', 'parPERC', 'parUZL', 'parTT', 'parCFMAX',
       'parCFR', 'parCWH', 'parBETAET']
CASES = [
    # name, T, B, nmul, warm_up, dynamic, n_par  (the first five: tests/test_hbv_adj_gpu.py)
    ('static', 120, 9, 4, 0, [], 12),
    ('d2_warm', 150, 7, 16, 40, D2, 13),          # ring form
    ('d2_nowarm', 100, 33, 8, 0, D2, 13),
    ('all_dynamic', 90, 5, 4, 20, ALL, 13),
    ('d1_twelve', 80, 6, 2, 10, ['parK1'], 12),
    ('nmul3', 70, 11, 3, 15, D2, 13),             # shared-memory nmul reduction
    ('nmul6_static', 60, 5, 6, 0, [], 12),
]
CASE = {c[0]: c for c in CASES}
COLS = ('prcp', 'tmean', 'pet')


class _NewtonStepForcing(torch.autograd.Function):
    """The oracle's implicit step (oracle/hbv_adj_oracle.py: _NewtonStep, the adjoint of
    hbv_adj.py:620-633) plus the gradient w.r.t. the forcings, dL/dclim = -lambda^T dG/dclim,
    by autograd through the residual (the rain/snow mask T < TT carries no gradient, as in rhs)."""

    @staticmethod
    def forward(ctx, theta, xt, clim, dt, bounds, mode, tol, max_updates, stats):
        from oracle import hbv_adj_oracle as AO
        x, J, n = AO.newton_solve(theta, xt, clim, dt, bounds, mode, tol, max_updates)
        if stats is not None:
            stats.append(n)
        with torch.enable_grad():
            th = theta.detach().requires_grad_(True)
            gg = AO.residual(x.detach(), th, xt.detach(), clim.detach(), dt, bounds)
            dGdp = AO.batch_jacobian(gg, th).detach()
        ctx.save_for_backward(J, dGdp, x.detach(), theta.detach(), xt.detach(), clim.detach())
        ctx.dt, ctx.bounds = dt, bounds
        return x.detach()

    @staticmethod
    def backward(ctx, dLdx):
        from oracle import hbv_adj_oracle as AO
        J, dGdp, x, theta, xt, clim = ctx.saved_tensors
        lam = torch.linalg.solve(J.transpose(1, 2), dLdx)          # [N,5]
        dLdp = -torch.bmm(lam.unsqueeze(1), dGdp).squeeze(1)
        dLdxt = lam / ctx.dt                                       # dG/dxt = -I/dt
        dLdclim = None
        if ctx.needs_input_grad[2]:
            with torch.enable_grad():
                cl = clim.detach().requires_grad_(True)
                gg = AO.residual(x, theta, xt, cl, ctx.dt, ctx.bounds)
                dLdclim, = torch.autograd.grad(gg, cl, grad_outputs=-lam)
        return dLdp, dLdxt, dLdclim, None, None, None, None, None, None


@contextlib.contextmanager
def _oracle_with_forcing_grad():
    """oracle.hbv_adj_oracle with its time loop (`integrate`) stepping through
    _NewtonStepForcing, so that x_phy.grad is filled by forward_adj's backward."""
    from oracle import hbv_adj_oracle as AO
    saved = AO._NewtonStep
    AO._NewtonStep = _NewtonStepForcing
    try:
        yield AO
    finally:
        AO._NewtonStep = saved


def test_oracle_forcing_gradient_matches_finite_difference():
    """CPU, float64: the oracle leg's d loss / d x_phy (-lambda^T dG/dclim, _NewtonStepForcing)
    equals central differences of the forward solve, warm-up rows included.  Newton is converged
    tightly so the differences are not Newton noise; an entry is probed only where the forward
    and backward one-sided differences agree (away from the min / clamp / rain-snow kinks)."""
    from oracle import hbv_adj_oracle as AO
    from oracle import hbv_oracle as O
    T, B, nmul, warm = 20, 2, 2, 5
    kw = dict(nmul=nmul, warm_up=warm, dynamic_params=D2, tol=1e-12, max_updates=50)
    x = O.synthetic_forcing(T, B, seed=61).double()
    p = torch.randn(T, B, 13 * nmul + 2, generator=torch.Generator().manual_seed(62)).double()
    w = torch.randn(T - warm, B, 1, generator=torch.Generator().manual_seed(63)).double()
    xg = x.clone().requires_grad_(True)
    with _oracle_with_forcing_grad() as AOF:
        (AOF.forward_adj(xg, p, **kw)['flow_sim'] * w).sum().backward()
    assert xg.grad.shape == x.shape and float(xg.grad[:warm].abs().max()) > 0

    def loss(xx):
        return float((AO.forward_adj(xx, p, **kw)['flow_sim'] * w).sum())

    eps = 1e-6
    l0 = loss(x)
    checked = {c: 0 for c in range(3)}
    gen = torch.Generator().manual_seed(64)
    for _ in range(36):
        t, b, c = (int(torch.randint(0, n, (1,), generator=gen)) for n in (T, B, 3))
        e = torch.zeros_like(x)
        e[t, b, c] = eps
        lp, lm = loss(x + e), loss(x - e)
        fwd, bwd = (lp - l0) / eps, (l0 - lm) / eps
        if abs(fwd - bwd) > 1e-4 * max(1.0, abs(fwd)):
            continue                                   # a kink within eps of this entry
        fd = (lp - lm) / (2 * eps)
        an = float(xg.grad[t, b, c])
        assert abs(fd - an) <= 1e-6 * max(1.0, abs(an)), (t, b, COLS[c], fd, an)
        checked[c] += 1
    assert all(n >= 3 for n in checked.values()), checked


def test_adj_bwd_rejects_a_call_without_outputs():
    """CPU: gdyn = NULL needs gdyn_zero_fill = 0 and at least one of gforcing / gstate_in (the
    arguments are checked before anything touches the device)."""
    import ctypes as C
    from hydrodl2_b200 import _build, _cabi
    _build.build()
    lib = _cabi.load()
    d = _cabi.HbvDesc()
    d.abi_version, d.variant = _cabi.ABI_VERSION, _cabi.VARIANT_ADJ
    io = _cabi.HbvAdjBwdIO()
    io.forcing = io.dyn = io.ysol = 256          # never dereferenced: the call is refused first
    assert lib.hbv_b200_adj_bwd(C.byref(d), C.byref(io), None) == -1          # HBV_E_NULL
    io.gforcing, io.gdyn_zero_fill = 256, 1
    assert lib.hbv_b200_adj_bwd(C.byref(d), C.byref(io), None) == -2          # HBV_E_SHAPE


# ------------------------------------------------------------------------------------------------
def _inputs(case, seed=21):
    from oracle import hbv_oracle as O
    name, T, B, nmul, warm, dyn, n_par = case
    x = O.synthetic_forcing(T, B, seed=seed)
    gen = torch.Generator().manual_seed(seed + 1)
    p = torch.randn(T, B, n_par * nmul + 2, generator=gen)
    cot = torch.randn(T - warm, B, 1, generator=gen)
    return x, p, cot


def _oracle(case, x, p, cot, routing=True, p_grad=True):
    name, T, B, nmul, warm, dyn, n_par = case
    x64 = x.double().requires_grad_(True)
    p64 = p.double().requires_grad_(p_grad)
    with _oracle_with_forcing_grad() as AOF:
        ref = AOF.forward_adj(x64, p64, nmul=nmul, warm_up=warm, dynamic_params=dyn, routing=routing)
        (ref['flow_sim'] * cot.double()).sum().backward()
    return ref['flow_sim'].detach(), x64.grad, p64.grad


def _model(case, routing=True, **cfg):
    import hydrodl2_b200 as hydrodl2
    name, T, B, nmul, warm, dyn, n_par = case
    M = hydrodl2.load_model('hbv_adj', ver_name='HbvAdj')
    return M(dict({'warm_up': warm, 'dynamic_params': {'HbvAdj': dyn}, 'nmul': nmul, 'routing': routing}, **cfg),
             device=torch.device('cuda:0'))


def _run(case, x, p, cot, routing=True, x_grad=True, p_grad=True, **cfg):
    dev = torch.device('cuda:0')
    m = _model(case, routing, **cfg)
    xg = x.to(dev).requires_grad_(x_grad)
    pg = p.to(dev).requires_grad_(p_grad)
    out = m({'x_phy': xg}, pg)
    (out['flow_sim'] * cot.to(dev)).sum().backward()
    return out['flow_sim'], xg.grad, pg.grad


def _check_forcing_grad(got, ref, what):
    assert got is not None and got.shape == ref.shape, what
    for c, col in enumerate(COLS):
        assert_close(got[..., c], ref[..., c], RTOL_GRAD, f'{what}: grad x_phy[{col}]')


@gpu
@pytest.mark.parametrize('case', CASES, ids=[c[0] for c in CASES])
def test_forcing_gradient_parity(case):
    x, p, cot = _inputs(case)
    flow, gx, gp = _run(case, x, p, cot)
    rflow, rgx, rgp = _oracle(case, x, p, cot)
    assert_close(flow, rflow, RTOL_FLUX, f'{case[0]}: flow_sim')
    assert_close(gp, rgp, RTOL_GRAD, f'{case[0]}: grad parameters')
    _check_forcing_grad(gx, rgx, case[0])
    warm = case[4]
    if warm > 0:
        # the warm-up is differentiable: its forcing rows carry gradient, and the right one
        assert float(gx[:warm].abs().max()) > 0
        _check_forcing_grad(gx[:warm], rgx[:warm], f'{case[0]} warm-up rows')


@gpu
@pytest.mark.parametrize('name', ['d2_warm', 'nmul3', 'static'])
def test_forcing_gradient_without_routing(name):
    case = CASE[name]
    x, p, cot = _inputs(case, seed=41)
    flow, gx, gp = _run(case, x, p, cot, routing=False)
    rflow, rgx, rgp = _oracle(case, x, p, cot, routing=False)
    assert_close(flow, rflow, RTOL_FLUX, f'{name}: flow_sim (no routing)')
    assert_close(gp, rgp, RTOL_GRAD, f'{name}: grad parameters (no routing)')
    _check_forcing_grad(gx, rgx, f'{name} (no routing)')


@gpu
def test_forcing_gradient_register_form_nmul16():
    """Option ring = 0 keeps the standard case (nmul 16, D2) on the register kernel, whose nmul sum
    is then a 16-lane shuffle inside 128-thread CTAs."""
    from hydrodl2_b200 import _cabi
    case = CASE['d2_warm']
    x, p, cot = _inputs(case)
    with _cabi.option('ring', 0):
        flow, gx, gp = _run(case, x, p, cot)
    rflow, rgx, rgp = _oracle(case, x, p, cot)
    assert_close(gp, rgp, RTOL_GRAD, 'register form: grad parameters')
    _check_forcing_grad(gx, rgx, 'register form')


@gpu
@pytest.mark.parametrize('name', ['d2_warm', 'nmul3', 'all_dynamic'])
def test_forcing_only(name):
    """Variational precipitation DA: parameters fixed, d loss / d x_phy wanted (the adjoint runs
    with gdyn = NULL; K4^T writes its routing gradient to a scratch)."""
    case = CASE[name]
    x, p, cot = _inputs(case, seed=51)
    flow, gx, gp = _run(case, x, p, cot, p_grad=False)
    assert gp is None
    rflow, rgx, _ = _oracle(case, x, p, cot, p_grad=False)
    assert_close(flow, rflow, RTOL_FLUX, f'{name}: flow_sim')
    _check_forcing_grad(gx, rgx, f'{name} forcing only')
    # and the same numbers as with the parameter gradient (the kernels share the step arithmetic)
    _, gx2, _ = _run(case, x, p, cot)
    assert_close(gx, gx2, 1e-6, f'{name}: forcing only vs with the parameter gradient')


@gpu
def test_forcing_only_allocates_no_parameter_plane():
    """At B = 2,000, T = 365, nmul 16 the [T, B, 210] parameter-gradient plane (613 MB) dominates
    the backward; with only x_phy requiring grad the backward's peak stays below one such plane."""
    case = ('big', 365, 2000, 16, 0, D2, 13)
    x, p, cot = _inputs(case, seed=81)
    dev = torch.device('cuda:0')
    plane = p.numel() * 4
    peaks = {}
    for p_grad in (False, True):
        m = _model(case)
        xg = x.to(dev).requires_grad_(True)
        pg = p.to(dev).requires_grad_(p_grad)
        loss = (m({'x_phy': xg}, pg)['flow_sim'] * cot.to(dev)).sum()
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        loss.backward()
        torch.cuda.synchronize()
        peaks[p_grad] = torch.cuda.max_memory_allocated() - base
        assert torch.isfinite(xg.grad).all() and float(xg.grad[..., 0].abs().max()) > 0
        del loss, xg, pg, m
    assert peaks[False] < plane, (peaks, plane)
    assert peaks[True] >= plane, (peaks, plane)      # (the measurement sees a plane when there is one)


@gpu
@pytest.mark.parametrize('name', ['d2_warm', 'static', 'nmul3'])
def test_parameter_gradient_unchanged_by_forcing_gradient(name):
    case = CASE[name]
    x, p, cot = _inputs(case, seed=91)
    _, _, gp0 = _run(case, x, p, cot, x_grad=False)
    gp0 = gp0.clone()
    _, gx, gp1 = _run(case, x, p, cot, x_grad=True)
    assert gx is not None
    assert torch.equal(gp0, gp1), float((gp0 - gp1).abs().max())


@gpu
@pytest.mark.parametrize('name', ['d2_warm', 'nmul3', 'nmul6_static'])
@pytest.mark.parametrize('p_grad', [True, False])
def test_forcing_gradient_deterministic(name, p_grad):
    case = CASE[name]
    x, p, cot = _inputs(case, seed=101)
    _, gx0, _ = _run(case, x, p, cot, p_grad=p_grad)
    _, gx1, _ = _run(case, x, p, cot, p_grad=p_grad)
    assert torch.equal(gx0, gx1)


@gpu
@pytest.mark.parametrize('name', ['d2_warm', 'all_dynamic'])
def test_forcing_gradient_column_mapping(name):
    """variables = [tmean, pet, prcp] plus an unused 4th column: each gradient lands in its own
    column and the unused one stays exactly 0; the oracle takes (prcp, tmean, pet)."""
    case = CASE[name]
    x, p, cot = _inputs(case, seed=111)
    perm = [1, 2, 0]                                   # model column k holds oracle column perm[k]
    x4 = torch.cat([x[..., perm], torch.randn(x.shape[:2] + (1,), generator=torch.Generator().manual_seed(112))], -1)
    flow, gx, gp = _run(case, x4, p, cot, variables=['tmean', 'pet', 'prcp', 'extra'])
    rflow, rgx, rgp = _oracle(case, x, p, cot)
    assert_close(flow, rflow, RTOL_FLUX, f'{name}: flow_sim (permuted columns)')
    assert_close(gp, rgp, RTOL_GRAD, f'{name}: grad parameters (permuted columns)')
    assert gx.shape == x4.shape
    _check_forcing_grad(gx[..., [2, 0, 1]], rgx, f'{name} permuted columns')
    assert float(gx[..., 3].abs().max()) == 0.0


# ------------------------------------------------------------------------------------------------
def _stream_inputs(T, B, nmul, seed):
    from oracle import hbv_oracle as O
    x = O.synthetic_forcing(T, B, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    p = torch.randn(1, B, 13 * nmul + 2, generator=g).repeat(T, 1, 1)     # static values: the same at every row
    for i in (0, 12):                                                        # the two dynamic blocks vary in time
        p[:, :, i * nmul:(i + 1) * nmul] = torch.randn(T, B, nmul, generator=g)
    return x.cuda(), p.cuda()


CHUNKS = (30, 7, 1)


@gpu
@pytest.mark.parametrize('nmul', [16, 4])
def test_cache_states_chunked_equals_one_shot(nmul):
    T, B = sum(CHUNKS), 13
    x, p = _stream_inputs(T, B, nmul, 121)
    case = ('stream', T, B, nmul, 0, D2, 13)
    with torch.no_grad():
        one_m = _model(case, routing=False)
        one = one_m({'x_phy': x}, p)['flow_sim']
        m = _model(case, routing=False, cache_states=True)
        parts, t0 = [], 0
        for n in CHUNKS:
            parts.append(m({'x_phy': x[t0:t0 + n]}, p[t0:t0 + n])['flow_sim'])
            t0 += n
    assert_close(torch.cat(parts), one, 1e-6, 'chunked cache_states: flow_sim')
    for name, a, b in zip(m.state_names, m.get_states(), one_m.get_states()):
        assert a.shape == (B, nmul)
        assert_close(a, b, 1e-6, f'cached state {name}', floor=STATE_FLOOR)


@gpu
def test_uh_carry_over_routed_equals_one_shot():
    T, B, nmul = sum(CHUNKS), 9, 16
    x, p = _stream_inputs(T, B, nmul, 131)
    case = ('stream', T, B, nmul, 0, D2, 13)
    with torch.no_grad():
        one = _model(case)({'x_phy': x}, p)['flow_sim']
        m = _model(case, cache_states=True, uh_carry_over=True)
        parts, t0 = [], 0
        for n in CHUNKS:
            parts.append(m({'x_phy': x[t0:t0 + n]}, p[t0:t0 + n])['flow_sim'])
            t0 += n
    assert_close(torch.cat(parts), one, 1e-6, 'uh_carry_over: routed flow_sim')
    # inference only: the routed history carries no gradient
    with pytest.raises(RuntimeError, match='uh_carry_over'):
        m({'x_phy': x[:5]}, p[:5].clone().requires_grad_(True))
    with pytest.raises(RuntimeError, match='uh_carry_over'):
        m({'x_phy': x[:5].clone().requires_grad_(True)}, p[:5])


@gpu
def test_load_states_round_trip_and_errors():
    T, B, nmul, split = 40, 6, 4, 25
    x, p = _stream_inputs(T, B, nmul, 141)
    case = ('stream', T, B, nmul, 0, D2, 13)
    a = _model(case, routing=False, cache_states=True)
    assert a.get_states() is None
    with torch.no_grad():
        a({'x_phy': x[:split]}, p[:split])
        b = _model(case, routing=False, cache_states=True)
        b.load_states(a.get_states())
        assert all(torch.equal(s, r) and not s.requires_grad for s, r in zip(b.states, a.get_states()))
        qa = a({'x_phy': x[split:]}, p[split:])['flow_sim']
        qb = b({'x_phy': x[split:]}, p[split:])['flow_sim']
    assert torch.equal(qa, qb)
    with pytest.raises(ValueError):
        b.load_states(list(a.get_states()))
    with pytest.raises(ValueError):
        b.load_states(a.get_states()[:4])
    with pytest.raises(ValueError):
        b.load_states(tuple(a.get_states()[:4]) + (1.0,))
    # cached states of another grid size are refused, not read out of bounds
    with pytest.raises(ValueError):
        b({'x_phy': x[:5, :3].contiguous()}, p[:5, :3].contiguous())
