"""Forward-mode AD cost: "forward only" against "forward + JVP" (torch.autograd.forward_ad), the
two alternating in one process.  Reports the median and min-max CUDA-event time of each library
call: K1 (hbv_fwd, the kernel family the dispatcher picks), K1t (hbv_tlm), K4 (route_fwd), K4t
(route_tlm) and the warm-up runs.

    python scripts/forward_ad_bench.py [--reps 5] [--out profiles/r04_forward_ad.json] [--only c2]

Shapes: C2 (`hbv`, dynamic [parBETA, parBETAET], nmul 16, 531 basins, 365 warm-up + 730 days),
the same model on the 22,500-basin shard, and the per-GPU hourly grid of BASELINE config 4
without routing (`hbv_2_hourly`, dynamic [parBETA, parK0, parBETAET], 2,500 units x 17,520 h).
Tangents: one random direction on every input (parameters and forcings)."""

from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch
import torch.autograd.forward_ad as fwAD

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _packed(B, T, warm):
    import hydrodl2_b200 as hydrodl2
    from oracle import hbv_oracle as O
    dev = torch.device('cuda')
    m = hydrodl2.load_model('hbv', ver_name='Hbv')({'warm_up': warm, 'nmul': 16,
                                                    'dynamic_params': {'Hbv': ['parBETA', 'parBETAET']}},
                                                   device=dev)
    g = torch.Generator(device=dev).manual_seed(1)
    x = O.synthetic_forcing(T, B, seed=2).to(dev)
    p = torch.randn(T, B, 13 * 16 + 2, device=dev, generator=g)
    vx = 0.1 * torch.randn(x.shape, device=dev, generator=g)
    vp = torch.randn(p.shape, device=dev, generator=g)
    return (lambda xx, pp: m({'x_phy': xx}, pp)), (x, p), (vx, vp)


def _hourly(B, T):
    import hydrodl2_b200 as hydrodl2
    from oracle import hbv_oracle as O
    dev = torch.device('cuda')
    dyn = ['parBETA', 'parK0', 'parBETAET']
    m = hydrodl2.load_model('hbv_2_hourly', ver_name='Hbv_2_hourly')(
        {'nmul': 16, 'routing': False, 'dynamic_params': {'Hbv_2_hourly': dyn}, 'state_series': False}, device=dev)
    m.use_distr_routing = False
    g = torch.Generator(device=dev).manual_seed(3)
    x = O.synthetic_forcing(T, B, seed=4, hourly=True).to(dev)
    p0 = torch.rand(T, B, len(dyn) * 16, device=dev, generator=g)
    p1 = torch.rand(B, 16 * 16, device=dev, generator=g)
    ac = torch.rand(B, device=dev, generator=g) * 5000
    el = torch.rand(B, device=dev, generator=g) * 3000
    v = tuple(0.1 * torch.randn(t.shape, device=dev, generator=g) for t in (x, p0, p1))
    return (lambda xx, q0, q1: m({'x_phy': xx, 'ac_all': ac, 'elev_all': el}, (q0, q1))), (x, p0, p1), v


CASES = {
    'c2': ('hbv D2, 531 basins x (365 + 730) days', lambda: _packed(531, 1095, 365)),
    'shard': ('hbv D2, 22,500 basins x (365 + 730) days', lambda: _packed(22500, 1095, 365)),
    'c4_hourly': ('hbv_2_hourly D3, 2,500 units x 17,520 h, no routing', lambda: _hourly(2500, 17520)),
}


def _collect(prof):
    return {k: [e0.elapsed_time(e1) for e0, e1 in v] for k, v in prof.items()}


def run_case(name, reps):
    from hydrodl2_b200 import ops
    what, make = CASES[name]
    fn, prim, tan = make()
    times = {'forward': {}, 'forward+jvp': {}}
    for it in range(reps + 1):
        for mode in ('forward', 'forward+jvp'):
            ops.PROFILE = {}
            with torch.no_grad():
                if mode == 'forward':
                    fn(*prim)
                else:
                    with fwAD.dual_level():
                        fn(*[fwAD.make_dual(p, t) for p, t in zip(prim, tan)])
            torch.cuda.synchronize()
            got = _collect(ops.PROFILE)
            ops.PROFILE = None
            if it == 0:
                continue          # first round: module load, allocator growth
            for k, v in got.items():
                times[mode].setdefault(k, []).extend(v)
    summary = {mode: {k: {'median_ms': statistics.median(v), 'min_ms': min(v), 'max_ms': max(v), 'n': len(v)}
                      for k, v in d.items()} for mode, d in times.items()}
    return {'case': what, 'reps': reps, **summary}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    ap.add_argument('--only', default=None)
    a = ap.parse_args()
    from hydrodl2_b200 import _build
    _build.build()
    props = torch.cuda.get_device_properties(0)
    res = {'gpu': props.name, 'torch': torch.__version__, 'cases': {}}
    for name in CASES:
        if a.only and name != a.only:
            continue
        res['cases'][name] = run_case(name, a.reps)
        print(json.dumps({name: res['cases'][name]}), flush=True)
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
