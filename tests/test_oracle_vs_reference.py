"""Where the unmodified reference is installed (the git-ignored baseline/_ref, laid down by
scripts/install_reference.py from a mhpi/hydrodl2 source checkout), pin the oracle against it
directly on fresh seeded cases — beyond the committed golden fixtures.  Skipped without it (the
fixtures in tests/golden/ carry the pin then).
"""

import os
import sys

import pytest
import torch

REF_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'baseline', '_ref')
pytestmark = pytest.mark.skipif(not os.path.isdir(os.path.join(REF_DIR, 'hydrodl2')),
                                reason='baseline/_ref not installed (scripts/install_reference.py)')

NMUL = 4


@pytest.fixture(scope='module')
def ref():
    os.environ.setdefault('CI', '1')          # licence prompt bypass of the reference's __init__
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import hydrodl2
    return hydrodl2


@pytest.mark.parametrize('model,cls,npar,dyn,warm', [
    ('hbv', 'Hbv', 13, ['parBETA', 'parBETAET'], 9),
    ('hbv', 'Hbv', 12, [], 0),
    ('hbv_1_1p', 'Hbv_1_1p', 14, ['parBETA', 'parK0', 'parBETAET'], 5),
    ('hbv_1_1p', 'Hbv_1_1p', 14, ['parFC', 'parTT', 'parC'], 0),
])
@pytest.mark.parametrize('seed', [101, 202])
def test_oracle_bit_exact_against_reference_packed(ref, model, cls, npar, dyn, warm, seed):
    from oracle import hbv_oracle as O
    T, B = 41, 6
    x = O.synthetic_forcing(T, B, seed=seed)
    p = torch.randn(T, B, npar * NMUL + 2, generator=torch.Generator().manual_seed(seed + 1))
    M = ref.load_model(model, ver_name=cls)
    m = M({'warm_up': warm, 'dynamic_params': {cls: dyn}, 'nmul': NMUL}, device=torch.device('cpu'))
    pr = p.clone().requires_grad_(True)
    torch.manual_seed(seed)
    out_ref = m({'x_phy': x}, pr)
    out_ref['streamflow'].sum().backward()

    po = p.clone().requires_grad_(True)
    out, _ = O.forward_packed(model, x, po, nmul=NMUL, warm_up=warm, dynamic_params=dyn)
    out['streamflow'].sum().backward()
    assert set(out) == set(out_ref)
    for k, v in out_ref.items():
        assert torch.equal(out[k], v.detach()), f'{model} {dyn}: {k} differs from the reference'
    assert torch.allclose(po.grad, pr.grad, rtol=1e-6, atol=1e-9), f'{model} {dyn}: gradient'


@pytest.mark.parametrize('routing', [False, True])
@pytest.mark.parametrize('seed', [303, 404])
def test_oracle_bit_exact_against_reference_hbv_2(ref, routing, seed):
    from oracle import hbv_oracle as O
    T, B = 33, 5
    dyn = ['parBETA', 'parK0', 'parBETAET']
    g = torch.Generator().manual_seed(seed)
    x = O.synthetic_forcing(T, B, seed=seed)
    n_sta = 13
    p0 = torch.rand(T, B, 3 * NMUL, generator=g)
    p1 = torch.rand(B, n_sta * NMUL + 2, generator=g)
    xd = {'x_phy': x, 'ac_all': torch.rand(B, generator=g) * 5000, 'elev_all': torch.rand(B, generator=g) * 3500}
    M = ref.load_model('hbv_2', ver_name='Hbv_2')
    m = M({'dynamic_params': {'Hbv_2': dyn}, 'nmul': NMUL, 'routing': routing}, device=torch.device('cpu'))
    a0, a1 = p0.clone().requires_grad_(True), p1.clone().requires_grad_(True)
    torch.manual_seed(seed)
    out_ref = m(xd, [a0, a1])
    out_ref['streamflow'].sum().backward()
    b0, b1 = p0.clone().requires_grad_(True), p1.clone().requires_grad_(True)
    out, _ = O.forward_split('hbv_2', xd, [b0, b1], nmul=NMUL, dynamic_params=dyn, routing=routing)
    out['streamflow'].sum().backward()
    for k, v in out_ref.items():
        assert torch.equal(out[k], v.detach()), f'hbv_2 routing={routing}: {k} differs from the reference'
    assert torch.allclose(b0.grad, a0.grad, rtol=1e-6, atol=1e-9)
    assert torch.allclose(b1.grad, a1.grad, rtol=1e-6, atol=1e-9)


def test_oracle_bit_exact_against_reference_hbv_2_hourly(ref):
    from oracle import hbv_oracle as O
    T, n_units, n_gages = 96, 6, 2
    dyn = ['parBETA', 'parK0', 'parBETAET']
    g = torch.Generator().manual_seed(505)
    x = O.synthetic_forcing(T, n_units, seed=505, hourly=True)
    p0 = torch.rand(T, n_units, 3 * NMUL, generator=g)
    p1 = torch.rand(n_units, 16 * NMUL, generator=g)
    topo = torch.zeros(n_gages, n_units)
    topo[0, :4] = 1
    topo[1, 2:] = 1                       # units 2, 3 drain to both gages (nested)
    p2 = torch.rand(int(topo.sum().item()), 3, generator=g)
    xd = {'x_phy': x, 'ac_all': torch.rand(n_units, generator=g) * 5000,
          'elev_all': torch.rand(n_units, generator=g) * 3500, 'outlet_topo': topo,
          'areas': torch.rand(n_units, generator=g) * 99 + 1}
    M = ref.load_model('hbv_2_hourly', ver_name='Hbv_2_hourly')
    m = M({'dynamic_params': {'Hbv_2_hourly': dyn}, 'nmul': NMUL}, device=torch.device('cpu'))
    a = [q.clone().requires_grad_(True) for q in (p0, p1, p2)]
    torch.manual_seed(505)
    out_ref = m(xd, a)
    out_ref['streamflow'].sum().backward()
    b = [q.clone().requires_grad_(True) for q in (p0, p1, p2)]
    out, _ = O.forward_split('hbv_2_hourly', xd, b, nmul=NMUL, dynamic_params=dyn)
    out['streamflow'].sum().backward()
    for k in ('Qs', 'streamflow'):
        assert torch.allclose(out[k], out_ref[k].detach(), rtol=1e-6, atol=1e-9), f'hourly: {k}'
    for gb, ga in zip(b, a):
        assert torch.allclose(gb.grad, ga.grad, rtol=1e-5, atol=1e-9)
