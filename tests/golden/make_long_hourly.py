"""Long-sequence fixture for BASELINE config 4: hbv_2_hourly, 17,520 hourly steps, fwd + bwd.

    python tests/golden/make_long_hourly.py        (~6 min of CPU; build container or GPU box)

The reference's own autograd over 17,520 unrolled steps is superlinear in T (CopySlices,
SURVEY.md §3c) and does not finish in reasonable time or memory, so the numbers come from the CPU
oracle (oracle/hbv_oracle.py — pinned bit-exact against the unmodified reference on the golden
cases incl. `hbv_2_hourly_d3`, tests/test_oracle_golden.py / test_oracle_vs_reference.py), run
once in float32 (the reference's arithmetic) and once in float64 (the arbiter of SURVEY §8 d6).
Inputs are regenerated from seeds by `inputs()` below (torch CPU generators are reproducible
across machines with the same torch build); only outputs are stored:
  Qs32 / Qs64          [T / QS_STRIDE, B]         unit runoff (x dt) at every QS_STRIDE-th step,
                                                  float32 / float64 evaluation
  S32 / S64            [5, B, nmul]               final storages
  gsta32 / gsta64      [B, 16 * nmul]             gradient w.r.t. the static parameter tensor
  gdyn32 / gdyn64      [len(rows), B, 3 * nmul]   gradient w.r.t. the dynamic tensor at `rows`
for the loss  sum(Qs * c)  with the seeded cotangent c of `inputs()`.  To keep the file under
1 MB, Qs64 and gdyn64 are stored as their float32 difference from Qs32 and gdyn32 (`save()`);
`load()` restores them to within 1e-12 of the float64 values, far below the float32-vs-float64
gap the tests measure.
"""

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

T, B, NMUL = 17520, 8, 16
DYN = ['parBETA', 'parK0', 'parBETAET']
ROW_STRIDE = 30
QS_STRIDE = 3
SEED = 4017520
PATH = os.path.join(HERE, 'hbv_2_hourly_long.npz')


def inputs(n_extra_units: int = 0):
    """Seeded inputs of the fixture: (x_dict, dyn [T, B, 48], sta [B, 256], cotangent [T, B, 1]).
    `n_extra_units` appends that many further units (own seed) after the fixture's B — the GPU
    test runs the 2,500-unit per-GPU grid of config 4 and compares the first B units."""
    from oracle.hbv_oracle import synthetic_forcing
    g = torch.Generator().manual_seed(SEED)
    x = synthetic_forcing(T, B, seed=SEED + 1, hourly=True)
    dyn = torch.rand(T, B, len(DYN) * NMUL, generator=g)
    sta = torch.rand(B, 16 * NMUL, generator=g)
    ac = torch.rand(B, generator=g) * 5000
    el = torch.rand(B, generator=g) * 3500
    cot = torch.rand(T, B, 1, generator=g)
    if n_extra_units:
        g2 = torch.Generator().manual_seed(SEED + 2)
        x = torch.cat([x, synthetic_forcing(T, n_extra_units, seed=SEED + 3, hourly=True)], dim=1)
        dyn = torch.cat([dyn, torch.rand(T, n_extra_units, len(DYN) * NMUL, generator=g2)], dim=1)
        sta = torch.cat([sta, torch.rand(n_extra_units, 16 * NMUL, generator=g2)], dim=0)
        ac = torch.cat([ac, torch.rand(n_extra_units, generator=g2) * 5000])
        el = torch.cat([el, torch.rand(n_extra_units, generator=g2) * 3500])
    return {'x_phy': x.contiguous(), 'ac_all': ac, 'elev_all': el}, dyn.contiguous(), sta.contiguous(), cot


def run(dtype):
    from oracle import hbv_oracle as O
    xd, dyn, sta, cot = inputs()
    p0 = dyn.clone().requires_grad_(True)
    p1 = sta.clone().requires_grad_(True)
    out, series = O.forward_split('hbv_2_hourly', xd, [p0, p1], nmul=NMUL, dynamic_params=DYN,
                                  use_distr_routing=False, dtype=dtype)
    (out['Qs'] * cot.to(out['Qs'].dtype)).sum().backward()
    S = torch.stack([s[-1] for s in series])
    rows = torch.arange(0, T, ROW_STRIDE)
    return out['Qs'][:, :, 0].detach(), S.detach(), p1.grad, p0.grad[rows], rows


def save(q32, q64, s32, s64, gs32, gs64, gd32, gd64, rows):
    """Numpy arrays of run(None) / run(torch.float64) -> PATH."""
    q32 = q32[::QS_STRIDE]
    dq = q64[::QS_STRIDE] - q32
    dg = gd64 - gd32
    np.savez_compressed(
        PATH, Qs32=q32, dQs64=dq.astype(np.float32), S32=s32, S64=s64, gsta32=gs32, gsta64=gs64,
        gdyn32=gd32, dgdyn64=dg.astype(np.float32), rows=rows,
        meta=np.array([T, B, NMUL, ROW_STRIDE, SEED, QS_STRIDE]))


def load():
    """-> {name: torch tensor} with the names of the module docstring, float64 results restored."""
    z = np.load(PATH)
    ref = {k: torch.from_numpy(z[k]) for k in z.files if k != 'meta'}
    ref['Qs64'] = ref['Qs32'].double() + ref.pop('dQs64').double()
    ref['gdyn64'] = ref['gdyn32'].double() + ref.pop('dgdyn64').double()
    return ref


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    q32, s32, gs32, gd32, rows = run(None)
    q64, s64, gs64, gd64, _ = run(torch.float64)
    save(q32.numpy(), q64.numpy(), s32.numpy(), s64.numpy(), gs32.numpy(), gs64.double().numpy(),
         gd32.numpy(), gd64.double().numpy(), rows.numpy())
    print(PATH, f'{os.path.getsize(PATH) / 1e6:.2f} MB')


if __name__ == '__main__':
    main()
