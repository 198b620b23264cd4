import sys, torch
sys.path.insert(0, 'tests'); sys.path.insert(0, '.')
import ctypes as C
import test_forward_ad_gpu as T_
from hydrodl2_b200 import _cabi as A, ops
DEV = T_.DEV
T, B, nmul = 50, 9, 4
x, p, vp, vx = T_._packed_inputs('hbv', T, B, nmul, seed=25)
m = T_._model('hbv', {'dynamic_params': {'Hbv': ['parBETA', 'parBETAET']}, 'nmul': nmul})
for dyn in (['parBETA', 'parBETAET'], []):
    spec = m._spec(dyn, routing=False)
    xx, pp, vpp, vxx = (t.to(DEV).contiguous() for t in (x, p, vp, vx))
    S0 = torch.full((5, B, nmul), 0.001, device=DEV)
    d = ops.make_desc(spec, T, B, 3, pp.shape[-1], 0); d.ckpt_interval = 0
    lib = A.load()
    f1 = torch.zeros((12, T, B), device=DEV); s1 = torch.zeros((5, B, nmul), device=DEV)
    ser1 = torch.zeros((5, T, B, nmul), device=DEV)
    io = A.HbvFwdIO(); io.forcing, io.dyn, io.state_in, io.state_out = xx.data_ptr(), pp.data_ptr(), S0.data_ptr(), s1.data_ptr()
    io.state_series = ser1.data_ptr()
    for f in range(11): io.flux[f] = f1[f].data_ptr()
    with A.option('lean', 0):
        A.check(lib.hbv_b200_fwd(C.byref(d), C.byref(io), ops._stream(DEV)), 'fwd')
    f2 = torch.zeros((12, T, B), device=DEV); f2t = torch.zeros_like(f2); s2 = torch.zeros_like(s1); s2t = torch.zeros_like(s1)
    tio = A.HbvTlmIO(); tio.forcing, tio.dyn, tio.state_in = xx.data_ptr(), pp.data_ptr(), S0.data_ptr()
    tio.forcing_t, tio.dyn_t = vxx.data_ptr(), vpp.data_ptr(); tio.state_out, tio.state_out_t = s2.data_ptr(), s2t.data_ptr()
    for f in range(11): tio.flux[f], tio.flux_t[f] = f2[f].data_ptr(), f2t[f].data_ptr()
    A.check(lib.hbv_b200_tlm(C.byref(d), C.byref(tio), ops._stream(DEV)), 'tlm')
    torch.cuda.synchronize()
    print('dyn', dyn, 'states equal', torch.equal(s1, s2))
    for f in range(11):
        dm = (f1[f] != f2[f])
        if dm.any():
            ts = dm.any(1).nonzero().flatten()
            print(' flux', f, 'ndiff', int(dm.sum()), 'first t', int(ts[0]), 'maxrel', ((f1[f]-f2[f]).abs().max()/f1[f].abs().max()).item())
