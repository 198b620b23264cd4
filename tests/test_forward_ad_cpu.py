"""CPU: argument validation of the forward-mode entry points (hbv_b200_tlm, hbv_b200_route_tlm),
and the reference leg of the GPU forward-mode tests — the oracle's own forward-AD JVP satisfies
the dot-product identity <w, J v> = <J^T w, v> against its reverse mode in float64."""

import ctypes as C

import pytest
import torch
import torch.autograd.forward_ad as fwAD

HBV_E_NULL, HBV_E_VARIANT, HBV_E_ABI = -1, -3, -6


@pytest.fixture(scope='module')
def lib():
    from hydrodl2_b200 import _build, _cabi
    _build.build()
    return _cabi.load()


def test_tlm_argument_validation(lib):
    from hydrodl2_b200 import _cabi as A
    d = A.HbvDesc()
    io = A.HbvTlmIO()
    assert lib.hbv_b200_tlm(None, None, None) == HBV_E_NULL
    assert lib.hbv_b200_tlm(C.byref(d), None, None) == HBV_E_NULL
    d.abi_version = A.ABI_VERSION
    d.variant = A.VARIANT_HBV
    assert lib.hbv_b200_tlm(C.byref(d), C.byref(io), None) == HBV_E_NULL      # no forcing / state_in
    io.forcing = io.state_in = io.dyn = 8
    d.abi_version = 999
    assert lib.hbv_b200_tlm(C.byref(d), C.byref(io), None) == HBV_E_ABI
    d.abi_version = A.ABI_VERSION
    d.variant = 9
    io.attrs = 8
    assert lib.hbv_b200_tlm(C.byref(d), C.byref(io), None) == HBV_E_VARIANT
    d.variant = A.VARIANT_ADJ
    assert lib.hbv_b200_tlm(C.byref(d), C.byref(io), None) == HBV_E_VARIANT
    d.variant = A.VARIANT_HBV2                                                 # needs attrs
    io.attrs = None
    assert lib.hbv_b200_tlm(C.byref(d), C.byref(io), None) == HBV_E_NULL
    assert lib.hbv_b200_last_error()


def test_route_tlm_argument_validation(lib):
    from hydrodl2_b200 import _cabi as A
    r = A.HbvRouteDesc()
    args = (8, None, 8, 16, 8, 16, 8, None, 8, 16, None, None, None)
    assert lib.hbv_b200_route_tlm(None, *args) == HBV_E_NULL
    r.abi_version = 999
    r.T, r.B, r.lenF, r.nser = 20, 4, 15, 4
    assert lib.hbv_b200_route_tlm(C.byref(r), *args) == HBV_E_ABI
    r.abi_version = A.ABI_VERSION
    no_tangent = (8, None, 8, 16, None, 16, 8, None, 8, 16, None, None, None)   # q_in_t NULL
    assert lib.hbv_b200_route_tlm(C.byref(r), *no_tangent) == HBV_E_NULL
    bfi_no_ws = (8, None, 8, 16, 8, 16, 8, None, 8, 16, 8, None, None)         # bfi_t without workspaces
    assert lib.hbv_b200_route_tlm(C.byref(r), *bfi_no_ws) == HBV_E_NULL


def test_abi_version_is_6(lib):
    from hydrodl2_b200 import _cabi as A
    assert A.ABI_VERSION == 6 and lib.hbv_b200_abi_version() == 6


def test_struct_size_matches_header():
    import os
    import subprocess
    import tempfile
    from hydrodl2_b200 import _cabi as A
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ('#include <stdio.h>\n#include "hbv_b200.h"\n'
            'int main(){printf("%zu\\n", sizeof(hbv_tlm_io_t));return 0;}')
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, 't.c')
        open(c, 'w').write(code)
        exe = os.path.join(td, 't')
        subprocess.check_call(['gcc', '-I', os.path.join(root, 'include'), c, '-o', exe])
        size = int(subprocess.check_output([exe]).split()[0])
    assert size == C.sizeof(A.HbvTlmIO)


@pytest.mark.parametrize('name', ['hbv', 'hbv_2'])
def test_oracle_forward_ad_dot_product_identity(name):
    """<w, J v> (oracle forward AD) == <J^T w, v> (oracle reverse mode) in float64, warm_up = 0,
    routing + BFI on: pins the reference leg of tests/test_forward_ad_gpu.py."""
    from oracle import hbv_oracle as O
    T, B, nmul = 40, 3, 2
    g = torch.Generator().manual_seed(41)
    x = O.synthetic_forcing(T, B, seed=42).double()
    dyn = ['parBETA', 'parBETAET'] if name == 'hbv' else ['parBETA', 'parK0']
    if name == 'hbv':
        prim = [x, torch.randn(T, B, 13 * nmul + 2, generator=g, dtype=torch.float64)]

        def f(xx, pp):
            return O.forward_packed('hbv', xx, pp, nmul=nmul, warm_up=0, dynamic_params=dyn)[0]
    else:
        xd = {'ac_all': torch.rand(B, generator=g, dtype=torch.float64) * 5000,
              'elev_all': torch.rand(B, generator=g, dtype=torch.float64) * 3000}
        prim = [x, torch.rand(T, B, 2 * nmul, generator=g, dtype=torch.float64),
                torch.rand(B, 14 * nmul + 2, generator=g, dtype=torch.float64)]

        def f(xx, q0, q1):
            return O.forward_split('hbv_2', {'x_phy': xx, **xd}, [q0, q1], nmul=nmul, dynamic_params=dyn,
                                   routing=True)[0]
    tan = [0.1 * torch.randn(p.shape, generator=g, dtype=torch.float64) for p in prim]
    with fwAD.dual_level():
        out = f(*[fwAD.make_dual(p, t) for p, t in zip(prim, tan)])
        jv = {k: fwAD.unpack_dual(v).tangent for k, v in out.items()}
    w = {k: torch.randn(v.shape, generator=g, dtype=torch.float64) for k, v in jv.items()}
    lhs = sum((w[k] * jv[k]).sum() for k in w)
    req = [p.clone().requires_grad_(True) for p in prim]
    out = f(*req)
    sum((w[k] * out[k]).sum() for k in w).backward()
    rhs = sum((p.grad * t).sum() for p, t in zip(req, tan))
    assert abs(lhs.item() - rhs.item()) <= 1e-10 * max(1.0, abs(lhs.item()))
