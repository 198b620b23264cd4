"""Print the measured parity margins (max-norm relative error) of the CUDA path against the
golden vectors of the unmodified reference.  GPU box:  python scripts/parity_report.py"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))
from conftest import STATE_FLOOR, load_golden, maxnorm_err  # noqa: E402


def state_err(a, b):
    """max-norm error of a storage tensor relative to max(||ref||, STATE_FLOOR) (conftest.py)."""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), STATE_FLOOR))
import test_parity_gpu as T  # noqa: E402


def main():
    dev = torch.device('cuda:0')
    worst = {'flux': 0.0, 'state': 0.0, 'grad': 0.0}
    for case in T.PACKED:
        g = load_golden(case)
        m, out, p = T._run_packed(g, dev)
        ef = max(maxnorm_err(out[k], ref) for k, ref in g['out'].items())
        kf = max(g['out'], key=lambda k: maxnorm_err(out[k], g['out'][k]))
        es = max(state_err(s, g['states'][n]) for n, s in zip(m.state_names, m.get_states()))
        loss = sum((out[k] * c.to(dev)).sum() for k, c in g['cot'].items())
        loss.backward()
        eg = maxnorm_err(p.grad, g['grad_parameters'])
        worst['flux'] = max(worst['flux'], ef)
        worst['state'] = max(worst['state'], es)
        worst['grad'] = max(worst['grad'], eg)
        print(f'{case:22s} flux {ef:.2e} ({kf})  state {es:.2e}  grad {eg:.2e}')
    for case in T.SPLIT:
        g = load_golden(case)
        m, out, params = T._run_split(g, dev)
        ef = max(maxnorm_err(out[k], ref) for k, ref in g['out'].items())
        kf = max(g['out'], key=lambda k: maxnorm_err(out[k], g['out'][k]))
        es = max(state_err(s, g['series'][n]) for n, s in zip(m.state_names, m._state_cache))
        loss = sum((out[k] * c.to(dev)).sum() for k, c in g['cot'].items())
        loss.backward()
        eg = max(maxnorm_err(p.grad, g['grad'][f'p{i}']) for i, p in enumerate(params))
        worst['flux'] = max(worst['flux'], ef)
        worst['state'] = max(worst['state'], es)
        worst['grad'] = max(worst['grad'], eg)
        print(f'{case:22s} flux {ef:.2e} ({kf})  state {es:.2e}  grad {eg:.2e}')
    print('worst', {k: f'{v:.2e}' for k, v in worst.items()}, ' tolerances: flux/state 1e-5, grad 1e-4')
    per_block(dev)
    full_size(dev)
    long_hourly(dev)


def per_block(dev):
    """Worst per-parameter-block gradient error (conftest.assert_grad_close) over the golden cases."""
    from conftest import assert_grad_close
    print('-- parameter gradients per parameter block (runs of nmul columns): worst relative error, block\n'
          '   (among blocks above 2e-3 of the tensor max-norm; smaller blocks are held to the fp32 noise floor, conftest.py)')
    for case in T.PACKED:
        g = load_golden(case)
        m, out, p = T._run_packed(g, dev)
        sum((out[k] * c.to(dev)).sum() for k, c in g['cot'].items()).backward()
        w = assert_grad_close(p.grad, g['grad_parameters'], case, int(g['meta'][2]))
        print(f'{case:22s} worst block {w[1]:2d}: {w[0]:.2e}')
    for case in T.SPLIT:
        g = load_golden(case)
        m, out, params = T._run_split(g, dev)
        sum((out[k] * c.to(dev)).sum() for k, c in g['cot'].items()).backward()
        ws = [assert_grad_close(q.grad, g['grad'][f'p{i}'], case, int(g['meta'][2]) if i < 2 else 1) for i, q in enumerate(params)]
        print(f'{case:22s} ' + '  '.join(f'p{i}: block {w[1]} {w[0]:.2e}' for i, w in enumerate(ws)))


def long_hourly(dev):
    """BASELINE config 4 at 17,520 steps (tests/test_long_hourly_gpu.py): margins against the fp32
    oracle and the float64 arbiter for every kernel family."""
    import test_long_hourly_gpu as L
    import make_long_hourly as G
    ref = G.load()
    fx = (G, ref) + tuple(G.inputs())
    print('-- hbv_2_hourly, 17,520 hourly steps, fwd + bwd: max-norm relative error vs the fp32 oracle | vs float64 '
          '(oracle fp32 vs float64 in brackets)')
    e = lambda a, b: maxnorm_err(a.double(), b.double())   # noqa: E731
    print(f"   oracle fp32 vs float64: Qs {e(ref['Qs32'], ref['Qs64']):.2e}  grad static {e(ref['gsta32'], ref['gsta64']):.2e}  "
          f"grad dynamic {e(ref['gdyn32'], ref['gdyn64']):.2e}")
    for n_units, ckpt, lean, what in L.CASES:
        qs, S, gsta, gdyn, fam = L._run(fx, n_units, ckpt, lean)
        print(f"   {what:62s} Qs {e(qs, ref['Qs32']):.2e} | {e(qs, ref['Qs64']):.2e}   grad static {e(gsta, ref['gsta32']):.2e} | "
              f"{e(gsta, ref['gsta64']):.2e}   grad dynamic {e(gdyn, ref['gdyn32']):.2e} | {e(gdyn, ref['gdyn64']):.2e}   "
              f"launches (lean, pipe) {fam}")
    from hydrodl2_b200 import _cabi
    _cabi.set_option('lean', -1)


def full_size(dev):
    """Margins against the CPU oracle at BASELINE sizes: C2 in full (K1s / K2s ring forms) and a
    48-basin slice of the 22,500-basin shards (K1s / K2s large-grid forms, K1d / K2d)."""
    import hydrodl2_b200 as hydrodl2
    from oracle import hbv_oracle as O
    D2 = ['parBETA', 'parBETAET']
    D14 = ['parBETA', 'parFC', 'parK0', 'parK1', 'parK2', 'parLP', 'parPERC', 'parUZL', 'parTT',
           'parCFMAX', 'parCFR', 'parCWH', 'parBETAET', 'parC']

    def run(name, cls, npar, dyn, T, B, warm, lo, nb, seed):
        g = torch.Generator(device=dev).manual_seed(seed)
        x = O.synthetic_forcing(T, B, seed=seed).to(dev) if B <= 4096 else None
        if x is None:
            import test_fullsize_gpu as F
            x, p = F._device_inputs(T, B, npar * 16 + 2, dev, seed)
        else:
            p = torch.randn(T, B, npar * 16 + 2, generator=g, device=dev)
        M = hydrodl2.load_model(name, ver_name=cls)
        m = M({'warm_up': warm, 'dynamic_params': {cls: dyn}, 'nmul': 16}, device=dev)
        pg = p.clone().requires_grad_(True)
        out = m({'x_phy': x}, pg)
        out['streamflow'].sum().backward()
        xs, ps = x[:, lo:lo + nb].cpu(), p[:, lo:lo + nb].cpu()
        pc = ps.clone().requires_grad_(True)
        ref, ref_states = O.forward_packed(name, xs, pc, nmul=16, warm_up=warm, dynamic_params=dyn)
        ref['streamflow'].sum().backward()
        ef = max(maxnorm_err(out[k][lo:lo + nb] if k == 'BFI' else out[k][:, lo:lo + nb], v) for k, v in ref.items())
        es = max(maxnorm_err(s[lo:lo + nb], r) for s, r in zip(m.get_states(), ref_states))
        eg = maxnorm_err(pg.grad[:, lo:lo + nb], pc.grad)
        print(f'{name:9s} {B:6d} x {T:4d} (warm-up {warm:3d}) vs oracle on basins [{lo}, {lo + nb}): '
              f'flux {ef:.2e}  state {es:.2e}  grad {eg:.2e}')

    run('hbv', 'Hbv', 13, D2, 1095, 531, 365, 0, 531, 20261017)
    run('hbv', 'Hbv', 13, D2, 730, 22500, 0, 11111, 128, 5)
    run('hbv_1_1p', 'Hbv_1_1p', 14, D14, 730, 22500, 0, 11111, 128, 5)


if __name__ == '__main__':
    main()
