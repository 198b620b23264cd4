"""GPU: forward-mode AD (torch.autograd.forward_ad) through the explicit HBV models — the
tangent-linear recurrence K1t and the routing tangent K4t.

The reference for every tangent is forward AD on the CPU oracle (oracle/hbv_oracle.py uses the
reference's own ops), in float32 and float64.  Adjoint consistency ties the new kernels to the
already-checked adjoint: <w, J v> from the JVP equals <J^T w, v> from the backward pass."""

import ctypes as C

import pytest
import torch
import torch.autograd.forward_ad as fwAD

from conftest import GRAD_BLOCK_FLOOR, RTOL_BY_KEY, STATE_FLOOR, arbiter_gate, assert_close

pytestmark = pytest.mark.gpu

DEV = torch.device('cuda:0')
RTOL_TAN = 1e-4          # the parameter-gradient bar
# The BFI tangent, 100 (num_t D - num den_t) / D^2, is a difference of two nearly equal terms
# wherever baseflow dominates (BFI ~ 100: num ~ den, num_t ~ den_t): the reference's own fp32
# tangent is 1.5e-4 to 1.6e-2 (relative) away from its fp64 one on these cases.  Like `excs`, it is
# held to the fp64 arbiter gate alone.
GATE_ONLY = set(RTOL_BY_KEY) | {'BFI'}
N_PACKED = {'hbv': 12, 'hbv_1_1p': 14}
CLS = {'hbv': 'Hbv', 'hbv_1_1p': 'Hbv_1_1p', 'hbv_2': 'Hbv_2', 'hbv_2_hourly': 'Hbv_2_hourly'}


def _model(name, cfg):
    import hydrodl2_b200 as hydrodl2
    m = hydrodl2.load_model(name, ver_name=CLS[name])(cfg, device=DEV)
    if name == 'hbv_2_hourly':
        m.use_distr_routing = False
    return m


def _tangent(v):
    t = fwAD.unpack_dual(v).tangent
    return torch.zeros_like(fwAD.unpack_dual(v).primal) if t is None else t


def _dual_tree(x, t):
    if isinstance(x, (tuple, list)):
        return type(x)(_dual_tree(a, b) for a, b in zip(x, t))
    if x is None:
        return None
    return x if t is None else fwAD.make_dual(x, t)


def _jvp(fn, primals, tangents):
    """-> (primal outputs, tangent outputs) of fn(*primals) with forward AD; nested dict / tuple
    outputs are flattened into {key: tensor}."""
    with fwAD.dual_level():
        out = fn(*_dual_tree(primals, tangents))
        flat = {}

        def walk(prefix, o):
            if isinstance(o, dict):
                for k, v in o.items():
                    walk(f'{prefix}{k}/', v)
            elif isinstance(o, (tuple, list)):
                for i, v in enumerate(o):
                    walk(f'{prefix}{i}/', v)
            elif isinstance(o, torch.Tensor):
                flat[prefix.rstrip('/')] = (fwAD.unpack_dual(o).primal.detach().clone(), _tangent(o).detach().clone())
        walk('', out)
    return {k: v[0] for k, v in flat.items()}, {k: v[1] for k, v in flat.items()}


def _to(tree, dev=None, dtype=None):
    if isinstance(tree, (tuple, list)):
        return type(tree)(_to(a, dev, dtype) for a in tree)
    if tree is None:
        return None
    return tree.to(device=dev if dev is not None else tree.device, dtype=dtype if dtype is not None else tree.dtype)


def _check_vs_oracle(new_t, ref32_t, ref64_t, what, keys=None, state_keys=()):
    """Every tangent series against the oracle's fp32 forward AD, with the rule of the parameter-
    gradient check (conftest.assert_grad_close):
        ||new - ref||_inf <= RTOL_TAN * ||ref||_inf + GRAD_BLOCK_FLOOR * (largest ||ref||_inf of the case)
    The second term matters for a series whose exact tangent is zero: where a flux is identically
    zero (the upper zone emptied by percolation every step, so Q1 = 0), the reference's fp32
    tangent is round-off residue (~1e-8, against ~1e-17 in fp64) and a relative error against it
    measures nothing.  Every series also passes the fp64 arbiter gate; the cancellation-limited
    series of RTOL_BY_KEY are held to the gate alone."""
    keys = keys if keys is not None else [k for k in ref32_t if k in new_t]
    assert keys, what
    gmax = max(ref32_t[k].detach().double().abs().max().item() for k in keys)
    for k in keys:
        a, r32, r64 = new_t[k].detach().cpu().reshape(ref32_t[k].shape), ref32_t[k], ref64_t[k]
        assert torch.isfinite(a).all(), f'{what}: tangent {k}: non-finite values'
        floor = STATE_FLOOR if k in state_keys else 0.0
        if k.split('/')[-1] not in GATE_ONLY:
            nb = max(r32.detach().double().abs().max().item(), floor)
            e = (a.double() - r32.detach().double()).abs().max().item()
            allowed = RTOL_TAN * nb + GRAD_BLOCK_FLOOR * gmax
            assert e <= allowed, (f'{what}: tangent {k}: error {e:.3e} > {allowed:.3e} (series max-norm '
                                  f'{nb:.3e}, largest of the case {gmax:.3e})')
        arbiter_gate(a, r32, r64, f'{what}: tangent {k} arbiter', floor=floor)


def _packed_inputs(name, T, B, nmul, seed, scale_x=0.1):
    from oracle import hbv_oracle as O
    x = O.synthetic_forcing(T, B, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    n = N_PACKED[name] + (1 if name == 'hbv' else 0)
    p = torch.randn(T, B, n * nmul + 2, generator=g)
    vp = torch.randn(p.shape, generator=g)
    vx = scale_x * torch.randn(x.shape, generator=g)
    return x, p, vp, vx


def _run_packed_case(name, T, B, nmul, warm, dyn, seed, dy_drop=0.0, tan_p=True, tan_x=True, muwts=False):
    from oracle import hbv_oracle as O
    x, p, vp, vx = _packed_inputs(name, T, B, nmul, seed)
    vp = vp if tan_p else None
    vx = vx if tan_x else None
    mu = vmu = None
    if muwts:
        g = torch.Generator().manual_seed(seed + 7)
        mu = torch.softmax(torch.randn(T - warm, B, nmul, generator=g), dim=-1)
        vmu = 0.1 * torch.randn(mu.shape, generator=g)
    cfg = {'warm_up': warm, 'dynamic_params': {CLS[name]: list(dyn)}, 'nmul': nmul, 'dy_drop': dy_drop}
    m = _model(name, cfg)

    def run_gpu(xx, pp, mm):
        torch.manual_seed(seed)
        xd = {'x_phy': xx}
        if mm is not None:
            xd['muwts'] = mm
        return m(xd, pp)
    _, new_t = _jvp(run_gpu, (x.to(DEV), p.to(DEV), _to(mu, DEV)),
                    (_to(vx, DEV), _to(vp, DEV), _to(vmu, DEV)))

    def run_ref(dtype):
        def f(xx, pp, mm):
            torch.manual_seed(seed)
            out, _ = O.forward_packed(name, xx, pp, nmul=nmul, warm_up=warm, dynamic_params=list(dyn),
                                      dy_drop=dy_drop, muwts=mm)
            return out
        return _jvp(f, _to((x, p, mu), dtype=dtype), _to((vx, vp, vmu), dtype=dtype))[1]
    return new_t, run_ref(torch.float32), run_ref(torch.float64)


# ---- oracle parity ------------------------------------------------------------------------------
def test_hbv_d2_warmup_routing_bfi():
    """`hbv`, dynamic [parBETA, parBETAET], warm-up 30, routing + BFI, tangents on `parameters`
    and `x_phy` (warm-up rows included: they reach the run through the warm-up's final states)."""
    new_t, r32, r64 = _run_packed_case('hbv', 90, 5, 4, 30, ['parBETA', 'parBETAET'], seed=101)
    _check_vs_oracle(new_t, r32, r64, 'hbv D2 warm-up 30')
    assert new_t['BFI'].abs().max() > 0 and new_t['streamflow'].abs().max() > 0


def test_warmup_rows_alone_carry_tangent():
    """A tangent on the warm-up's static row (parameters[warm_up - 1]) alone changes the run."""
    from oracle import hbv_oracle as O
    T, B, nmul, warm = 60, 3, 4, 20
    x, p, vp, _ = _packed_inputs('hbv', T, B, nmul, seed=5)
    vp = torch.zeros_like(vp)
    vp[warm - 1] = torch.randn(vp.shape[1:], generator=torch.Generator().manual_seed(3))
    m = _model('hbv', {'warm_up': warm, 'dynamic_params': {'Hbv': ['parBETA', 'parBETAET']}, 'nmul': nmul})
    _, new_t = _jvp(lambda xx, pp: m({'x_phy': xx}, pp), (x.to(DEV), p.to(DEV)), (None, vp.to(DEV)))

    def ref(dtype):
        f = (lambda xx, pp: O.forward_packed('hbv', xx, pp, nmul=nmul, warm_up=warm,
                                             dynamic_params=['parBETA', 'parBETAET'])[0])
        return _jvp(f, _to((x, p), dtype=dtype), (None, vp.to(dtype)))[1]
    r32, r64 = ref(torch.float32), ref(torch.float64)
    assert r64['streamflow_no_rout'].abs().max() > 0
    _check_vs_oracle(new_t, r32, r64, 'warm-up row only')


def test_hbv_1_1p_three_dynamic_dropout():
    new_t, r32, r64 = _run_packed_case('hbv_1_1p', 70, 6, 4, 10, ['parBETA', 'parK0', 'parBETAET'],
                                       seed=202, dy_drop=0.5)
    _check_vs_oracle(new_t, r32, r64, 'hbv_1_1p D3 dropout')


def test_hbv_static_nmul3():
    new_t, r32, r64 = _run_packed_case('hbv', 60, 7, 3, 0, [], seed=303)
    _check_vs_oracle(new_t, r32, r64, 'hbv static nmul 3')


def test_time_varying_muwts_tangent():
    new_t, r32, r64 = _run_packed_case('hbv', 50, 4, 4, 0, ['parBETA', 'parBETAET'], seed=404, muwts=True)
    _check_vs_oracle(new_t, r32, r64, 'hbv muwts')


def test_tangent_on_forcing_only():
    new_t, r32, r64 = _run_packed_case('hbv', 60, 5, 4, 15, ['parBETA', 'parBETAET'], seed=505, tan_p=False)
    _check_vs_oracle(new_t, r32, r64, 'x_phy only')


def _split_inputs(name, T, B, nmul, dyn, routing, seed):
    from oracle import hbv_oracle as O
    hourly = name == 'hbv_2_hourly'
    x = O.synthetic_forcing(T, B, seed=seed, hourly=hourly)
    g = torch.Generator().manual_seed(seed + 1)
    n = 19 if hourly else 16
    p0 = torch.rand(T, B, len(dyn) * nmul, generator=g)
    p1 = torch.rand(B, (n - len(dyn)) * nmul + (2 if routing else 0), generator=g)
    ac = torch.rand(B, generator=g) * 5000
    el = torch.rand(B, generator=g) * 3000
    v0 = 0.1 * torch.randn(p0.shape, generator=g)
    v1 = 0.1 * torch.randn(p1.shape, generator=g)
    vx = 0.1 * torch.randn(x.shape, generator=g)
    return x, p0, p1, ac, el, v0, v1, vx


def _run_split_case(name, T, B, nmul, dyn, routing, seed, states=False):
    from oracle import hbv_oracle as O
    x, p0, p1, ac, el, v0, v1, vx = _split_inputs(name, T, B, nmul, dyn, routing, seed)
    g = torch.Generator().manual_seed(seed + 9)
    S0 = tuple(0.5 + torch.rand(B, nmul, generator=g) for _ in range(5)) if states else None
    vS = tuple(0.1 * torch.randn(B, nmul, generator=g) for _ in range(5)) if states else None
    cfg = {'dynamic_params': {CLS[name]: list(dyn)}, 'nmul': nmul, 'routing': routing}
    m = _model(name, cfg)

    def run_gpu(xx, q0, q1, ss):
        xd = {'x_phy': xx, 'ac_all': ac.to(DEV), 'elev_all': el.to(DEV)}
        out = m(xd, (q0, q1), states=ss) if ss is not None else m(xd, (q0, q1))
        return {'out': out, 'series': m.get_states() if name == 'hbv_2_hourly' else m._state_cache}
    _, new_t = _jvp(run_gpu, (x.to(DEV), p0.to(DEV), p1.to(DEV), _to(S0, DEV)),
                    (vx.to(DEV), v0.to(DEV), v1.to(DEV), _to(vS, DEV)))

    def run_ref(dtype):
        def f(xx, q0, q1, ss):
            xd = {'x_phy': xx, 'ac_all': ac.to(dtype), 'elev_all': el.to(dtype)}
            out, series = O.forward_split(name, xd, [q0, q1], nmul=nmul, dynamic_params=list(dyn),
                                          routing=routing, states=ss, use_distr_routing=False)
            return {'out': out, 'series': series}
        return _jvp(f, _to((x, p0, p1, S0), dtype=dtype), _to((vx, v0, v1, vS), dtype=dtype))[1]
    return new_t, run_ref(torch.float32), run_ref(torch.float64)


def test_hbv_2_routing_state_series():
    new_t, r32, r64 = _run_split_case('hbv_2', 60, 5, 4, ['parBETA', 'parK0', 'parBETAET'], True, seed=606)
    keys = [k for k in r32 if k in new_t]
    state_keys = [k for k in keys if k.startswith('series')]
    assert len(state_keys) == 5
    _check_vs_oracle(new_t, r32, r64, 'hbv_2 routing + series', keys=keys, state_keys=state_keys)


def test_hbv_2_hourly_qs():
    new_t, r32, r64 = _run_split_case('hbv_2_hourly', 96, 4, 4, ['parBETA', 'parK0', 'parBETAET'], False, seed=707)
    _check_vs_oracle(new_t, r32, r64, 'hbv_2_hourly Qs', keys=['out/Qs'])


def test_initial_state_tangent_hourly_states_argument():
    new_t, r32, r64 = _run_split_case('hbv_2_hourly', 72, 4, 4, ['parBETA'], False, seed=808, states=True)
    keys = ['out/Qs'] + [f'series/{i}' for i in range(5)]
    _check_vs_oracle(new_t, r32, r64, 'hbv_2_hourly states=', keys=keys, state_keys=keys[1:])


def test_initial_state_tangent_packed_seam():
    """`_PBM` seam of the packed model: descaled parameter dict + states in, states out."""
    from oracle import hbv_oracle as O
    T, B, nmul = 40, 4, 4
    m = _model('hbv', {'dynamic_params': {'Hbv': []}, 'nmul': nmul})
    x = O.synthetic_forcing(T, B, seed=9)
    g = torch.Generator().manual_seed(10)
    names = list(m.parameter_bounds.keys())
    v = O.variant('hbv', names)
    prm = {k: (torch.rand(T, B, nmul, generator=g) * (hi - lo) + lo) for k, (lo, hi) in v.bounds.items()}
    S0 = tuple(0.5 + torch.rand(B, nmul, generator=g) for _ in range(5))
    vS = tuple(0.1 * torch.randn(B, nmul, generator=g) for _ in range(5))
    route = {'route_a': torch.rand(B, generator=g) * 2.9, 'route_b': torch.rand(B, generator=g) * 6.5}
    m.routing_param_dict = {k: t.to(DEV) for k, t in route.items()}

    def gpu(ss):
        fl, st = m._PBM(x.to(DEV), ss, {k: t.to(DEV) for k, t in prm.items()})
        return {'flux': fl, 'states': st}
    _, new_t = _jvp(gpu, (_to(S0, DEV),), (_to(vS, DEV),))

    def ref(dtype):
        def f(ss):
            fl, st, _ = O.run_pbm(v, x.to(dtype), ss, {k: t.to(dtype) for k, t in prm.items()}, nmul=nmul,
                                  routing=True, route={k: t.to(dtype) for k, t in route.items()})
            return {'flux': fl, 'states': st}
        return _jvp(f, (_to(S0, dtype=dtype),), (_to(vS, dtype=dtype),))[1]
    r32, r64 = ref(torch.float32), ref(torch.float64)
    keys = ['flux/streamflow', 'flux/streamflow_no_rout', 'flux/SWE', 'flux/recharge'] + [f'states/{i}' for i in range(5)]
    _check_vs_oracle(new_t, r32, r64, '_PBM states', keys=keys, state_keys=keys[4:])


# ---- adjoint consistency ------------------------------------------------------------------------
def _dot_identity(fn, primals, tangents, seed):
    """<w, J v> (forward mode) against <J^T w, v> (reverse mode), both in float64 from the fp32
    results, relative to sum |w| |J v|."""
    prim, jv = _jvp(fn, primals, tangents)
    g = torch.Generator().manual_seed(seed)
    w = {k: torch.randn(v.shape, generator=g).to(v.device) for k, v in prim.items()}
    lhs = sum((w[k].double() * jv[k].double()).sum() for k in w)
    scale = sum((w[k].double() * jv[k].double()).abs().sum() for k in w)
    req = [p.detach().clone().requires_grad_(True) if t is not None else p for p, t in zip(primals, tangents)]
    out = fn(*req)
    flat = {}

    def walk(prefix, o):
        if isinstance(o, dict):
            for k, v in o.items():
                walk(f'{prefix}{k}', v)
        elif isinstance(o, torch.Tensor):
            flat[prefix] = o
    walk('', out)
    loss = sum((w[k] * flat[k]).sum() for k in w if flat[k].requires_grad)
    loss.backward()
    rhs = sum((p.grad.double() * t.double()).sum() for p, t in zip(req, tangents) if t is not None)
    err = abs(lhs.item() - rhs.item()) / scale.item()
    assert err <= 1e-5, f'<w, Jv> = {lhs.item():.8e} vs <J^T w, v> = {rhs.item():.8e}: rel {err:.2e}'


def test_adjoint_consistency_packed_routing():
    x, p, vp, vx = _packed_inputs('hbv', 80, 6, 4, seed=11)
    m = _model('hbv', {'warm_up': 0, 'dynamic_params': {'Hbv': ['parBETA', 'parBETAET']}, 'nmul': 4})
    _dot_identity(lambda xx, pp: m({'x_phy': xx}, pp), (x.to(DEV), p.to(DEV)), (vx.to(DEV), vp.to(DEV)), 12)


def test_adjoint_consistency_hbv_2_routing():
    x, p0, p1, ac, el, v0, v1, vx = _split_inputs('hbv_2', 60, 5, 4, ['parBETA', 'parK0'], True, seed=13)
    m = _model('hbv_2', {'dynamic_params': {'Hbv_2': ['parBETA', 'parK0']}, 'nmul': 4, 'routing': True})
    xd = {'ac_all': ac.to(DEV), 'elev_all': el.to(DEV)}
    _dot_identity(lambda xx, q0, q1: m({'x_phy': xx, **xd}, (q0, q1)),
                  (x.to(DEV), p0.to(DEV), p1.to(DEV)), (vx.to(DEV), v0.to(DEV), v1.to(DEV)), 14)


def test_adjoint_consistency_tangent_after_warmup():
    """With a warm-up, tangents only on rows >= warm_up (the rows the reverse mode differentiates)."""
    x, p, vp, vx = _packed_inputs('hbv_1_1p', 70, 5, 4, seed=15)
    warm = 20
    vp[:warm] = 0
    m = _model('hbv_1_1p', {'warm_up': warm, 'dynamic_params': {'Hbv_1_1p': ['parBETA', 'parK0', 'parBETAET']},
                            'nmul': 4})
    _dot_identity(lambda pp: m({'x_phy': x.to(DEV)}, pp), (p.to(DEV),), (vp.to(DEV),), 16)


# ---- properties -------------------------------------------------------------------------------
def _packed_jvp(vp, vx, seed=21, dyn=('parBETA', 'parBETAET'), warm=10, p=None, x=None):
    x0, p0, _, _ = _packed_inputs('hbv', 60, 5, 4, seed=seed)
    x = x0 if x is None else x
    p = p0 if p is None else p
    m = _model('hbv', {'warm_up': warm, 'dynamic_params': {'Hbv': list(dyn)}, 'nmul': 4})
    return _jvp(lambda xx, pp: m({'x_phy': xx}, pp), (x.to(DEV), p.to(DEV)), (_to(vx, DEV), _to(vp, DEV)))


def test_zero_tangent_gives_exact_zero():
    _, _, vp, vx = _packed_inputs('hbv', 60, 5, 4, seed=21)
    _, t = _packed_jvp(torch.zeros_like(vp), torch.zeros_like(vx))
    for k, v in t.items():
        assert torch.count_nonzero(v) == 0, k


def test_linearity_and_determinism():
    _, _, vp, vx = _packed_inputs('hbv', 60, 5, 4, seed=22)
    g = torch.Generator().manual_seed(23)
    vp2, vx2 = torch.randn(vp.shape, generator=g), 0.1 * torch.randn(vx.shape, generator=g)
    _, t1 = _packed_jvp(vp, vx)
    _, t1b = _packed_jvp(vp, vx)
    _, t2x = _packed_jvp(2 * vp, 2 * vx)
    _, t2 = _packed_jvp(vp2, vx2)
    _, t12 = _packed_jvp(vp + vp2, vx + vx2)
    for k in t1:
        assert torch.equal(t1[k], t1b[k]), f'{k}: two runs differ'
        assert torch.equal(t2x[k], 2 * t1[k]), f'{k}: jvp(2v) != 2 jvp(v)'
        # (BFI: cancellation-limited, see GATE_ONLY — fp32 rounding of num_t, den_t is amplified)
        assert_close(t12[k], t1[k] + t2[k], 1e-4 if k == 'BFI' else 1e-6,
                     f'{k}: jvp(v1 + v2) vs jvp(v1) + jvp(v2)')


def test_dual_call_primal_bit_identical():
    x, p, vp, vx = _packed_inputs('hbv', 60, 5, 4, seed=24)
    prim, _ = _packed_jvp(vp, vx, p=p, x=x)
    m = _model('hbv', {'warm_up': 10, 'dynamic_params': {'Hbv': ['parBETA', 'parBETAET']}, 'nmul': 4})
    with torch.no_grad():
        plain = m({'x_phy': x.to(DEV)}, p.to(DEV))
    for k in plain:
        assert torch.equal(prim[k], plain[k]), k


@pytest.mark.parametrize('drop', [False, True])
def test_k1t_primal_outputs_equal_generic_k1(drop):
    """The optional primal outputs of hbv_b200_tlm equal the generic K1's bit for bit."""
    from hydrodl2_b200 import _cabi as A
    from hydrodl2_b200 import ops
    T, B, nmul = 50, 9, 4
    x, p, vp, vx = _packed_inputs('hbv', T, B, nmul, seed=25)
    m = _model('hbv', {'dynamic_params': {'Hbv': ['parBETA', 'parBETAET']}, 'nmul': nmul})
    spec = m._spec(['parBETA', 'parBETAET'], routing=False)
    x, p, vp, vx = (t.to(DEV).contiguous() for t in (x, p, vp, vx))
    S0 = torch.full((5, B, nmul), 0.001, device=DEV)
    drop_t = (torch.arange(13 * B, device=DEV).view(13, B) % 2).to(torch.uint8) if drop else None
    d = ops.make_desc(spec, T, B, 3, p.shape[-1], 0)
    d.ckpt_interval = 0
    lib = A.load()
    flux1 = torch.zeros((12, T, B), device=DEV)
    s1 = torch.zeros((5, B, nmul), device=DEV)
    io = A.HbvFwdIO()
    io.forcing, io.dyn, io.drop, io.state_in, io.state_out = x.data_ptr(), p.data_ptr(), ops._ptr(drop_t), S0.data_ptr(), s1.data_ptr()
    for f in range(11):
        io.flux[f] = flux1[f].data_ptr()
    with A.option('lean', 0):
        A.check(lib.hbv_b200_fwd(C.byref(d), C.byref(io), ops._stream(DEV)), 'fwd')
    flux2, flux2t = torch.zeros((12, T, B), device=DEV), torch.zeros((12, T, B), device=DEV)
    s2, s2t = torch.zeros((5, B, nmul), device=DEV), torch.zeros((5, B, nmul), device=DEV)
    tio = A.HbvTlmIO()
    tio.forcing, tio.dyn, tio.drop, tio.state_in = x.data_ptr(), p.data_ptr(), ops._ptr(drop_t), S0.data_ptr()
    tio.forcing_t, tio.dyn_t = vx.data_ptr(), vp.data_ptr()
    tio.state_out, tio.state_out_t = s2.data_ptr(), s2t.data_ptr()
    for f in range(11):
        tio.flux[f], tio.flux_t[f] = flux2[f].data_ptr(), flux2t[f].data_ptr()
    A.check(lib.hbv_b200_tlm(C.byref(d), C.byref(tio), ops._stream(DEV)), 'tlm')
    torch.cuda.synchronize()
    assert torch.equal(flux1, flux2)
    assert torch.equal(s1, s2)
    assert flux2t.abs().max() > 0


def test_reverse_mode_unaffected_by_duals():
    x, p, vp, vx = _packed_inputs('hbv', 60, 5, 4, seed=26)
    m = _model('hbv', {'warm_up': 10, 'dynamic_params': {'Hbv': ['parBETA', 'parBETAET']}, 'nmul': 4})
    g = torch.Generator().manual_seed(27)
    w = torch.randn(50, 5, 1, generator=g).to(DEV)
    pa = p.to(DEV).requires_grad_(True)
    xa = x.to(DEV).requires_grad_(True)
    (m({'x_phy': xa}, pa)['streamflow'] * w).sum().backward()
    pb = p.to(DEV).requires_grad_(True)
    xb = x.to(DEV).requires_grad_(True)
    with fwAD.dual_level():
        out = m({'x_phy': fwAD.make_dual(xb, vx.to(DEV))}, fwAD.make_dual(pb, vp.to(DEV)))
        (fwAD.unpack_dual(out['streamflow']).primal * w).sum().backward()
    assert torch.equal(pa.grad, pb.grad)
    assert torch.equal(xa.grad, xb.grad)


# ---- refusals -----------------------------------------------------------------------------------
def test_refusals():
    from hydrodl2_b200.routing import unit_routing
    from hydrodl2_b200 import ops
    x, p, vp, vx = _packed_inputs('hbv', 40, 3, 2, seed=31)
    xd, pd = x.to(DEV), p.to(DEV)
    with fwAD.dual_level():
        dual_p = fwAD.make_dual(pd, vp.to(DEV))
        # uh_carry_over (the routed history is detached)
        m = _model('hbv', {'dynamic_params': {'Hbv': []}, 'nmul': 2, 'cache_states': True, 'uh_carry_over': True})
        with pytest.raises(NotImplementedError, match='uh_carry_over'):
            m({'x_phy': xd}, dual_p)
        # initialize=True of the split models (and so Hbv_2_mts)
        _, p0, p1, ac, el, v0, v1, _ = _split_inputs('hbv_2', 40, 3, 2, [], False, seed=32)
        m2 = _model('hbv_2', {'dynamic_params': {'Hbv_2': []}, 'nmul': 2})
        m2.initialize = True
        with pytest.raises(NotImplementedError, match='initialize'):
            m2({'x_phy': xd, 'ac_all': ac.to(DEV), 'elev_all': el.to(DEV)},
               (None, fwAD.make_dual(p1.to(DEV), v1.to(DEV))))
        # a tangent on the attributes
        m2.initialize = False
        with pytest.raises(NotImplementedError, match='attributes'):
            m2({'x_phy': xd, 'ac_all': fwAD.make_dual(ac.to(DEV), torch.ones(3, device=DEV)),
                'elev_all': el.to(DEV)}, (None, p1.to(DEV)))
        # Hbv_2_mts
        from hydrodl2_b200.models.hbv.hbv_2_mts import Hbv_2_mts
        hi = {'dynamic_params': {'Hbv_2_hourly': []}, 'nmul': 2, 'train_spatial_chunk_size': 8,
              'simulate_spatial_chunk_size': 8, 'simulate_temporal_chunk_size': 8, 'train_warmup': 0}
        mts = Hbv_2_mts({'dynamic_params': {'Hbv_2': []}, 'nmul': 2}, hi, device=DEV)
        with pytest.raises(NotImplementedError, match='Hbv_2_mts'):
            mts({'areas': torch.ones(3)}, ((None, fwAD.make_dual(p1.to(DEV), v1.to(DEV))), (None, p1.to(DEV))))
        # pair routing / the long per-unit UH (K4')
        q = fwAD.make_dual(torch.rand(40, 3, device=DEV), torch.ones(40, 3, device=DEV))
        with pytest.raises(NotImplementedError, match='pair routing'):
            unit_routing(q, torch.rand(3, 2, device=DEV), 72, ((0, 5.0), (0, 12.0)))
        # HbvAdj (implicit scheme)
        import hydrodl2_b200 as hydrodl2
        ma = hydrodl2.load_model('hbv_adj', ver_name='HbvAdj')({'dynamic_params': {'HbvAdj': []}, 'nmul': 2,
                                                                'warm_up': 0}, device=DEV)
        with pytest.raises(NotImplementedError, match='HbvAdj'):
            ma({'x_phy': xd}, dual_p)
    assert ops.is_dual(xd) is False
