#!/usr/bin/env python
"""K3^T (the HbvAdj adjoint) with and without the forcing gradient, at the C5 shape (GPU box):

    python scripts/adj_forcing_bench.py [--reps 30] [--out FILE]

10,000 basins x 730 days, nmul 16, dynamic [parBETA, parBETAET] — the inputs of
scripts/bench_configs.run_c5.  Three backward modes over one forward graph each:
  off           parameters require grad, x_phy does not (the training step as before)
  on            both require grad: K3^T also writes d loss / d x_phy
  forcing_only  only x_phy requires grad: K3^T runs with gdyn = NULL, no parameter-gradient plane
K3^T time comes from CUDA events around each adjoint call (ops.PROFILE); the modes alternate
within one process, `reps` backward passes each after 3 untimed ones.  The [T, B, 210] plane
(6.1 GB) does not fit the 126 MB L2, so no pass reads a warm cache of it.  Peak memory is the
increase of torch.cuda.max_memory_allocated over one backward with the clean-plane cache off (so
a mode that needs a plane allocates it inside the measured window).  Prints one JSON object.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'scripts'))

import torch  # noqa: E402

from bench_configs import NMUL, forcing  # noqa: E402

MODES = ('off', 'on', 'forcing_only')


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout
        line = q.strip().splitlines()[torch.cuda.current_device()]
        name, power, clk = (s.strip() for s in line.split(','))
        return {'name': name, 'power_limit': power, 'max_sm_clock': clk}
    except Exception as e:             # (the torch name is still recorded)
        return {'name': torch.cuda.get_device_name(), 'power_limit': f'not read: {e}'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=30)
    ap.add_argument('--B', type=int, default=10000)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('adj_forcing_bench: needs a CUDA device (nothing is timed on the CPU)')
    import hydrodl2_b200 as hydrodl2
    from hydrodl2_b200 import ops
    dev = torch.device('cuda:0')
    T, B = 730, args.B
    dyn = ['parBETA', 'parBETAET']
    x0 = forcing(T, B, dev, 50)
    p0 = torch.randn(T, B, 13 * NMUL + 2, generator=torch.Generator(device=dev).manual_seed(5), device=dev)
    M = hydrodl2.load_model('hbv_adj', ver_name='HbvAdj')
    m = M({'warm_up': 0, 'dynamic_params': {'HbvAdj': dyn}, 'nmul': NMUL}, device=dev)

    graphs = {}
    for mode in MODES:
        x = x0.clone().requires_grad_(mode != 'off')
        p = p0.clone().requires_grad_(mode != 'forcing_only')
        loss = m({'x_phy': x}, p)['flow_sim'].sum()
        graphs[mode] = (loss, x, p)

    def backward(mode):
        loss, x, p = graphs[mode]
        x.grad = p.grad = None
        loss.backward(retain_graph=True)

    def release(mode):
        # (drop the gradients at once: the plane goes back to the clean-plane cache, so every
        # pass of 'off' and 'on' runs on a kept plane, as consecutive training steps do)
        graphs[mode][1].grad = graphs[mode][2].grad = None

    # peak memory of one backward per mode, every buffer allocated inside the window
    reuse = ops.REUSE_GRAD_PLANE
    ops.REUSE_GRAD_PLANE = False
    ops._PLANES.clear()
    peak = {}
    for mode in MODES:
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        backward(mode)
        torch.cuda.synchronize()
        peak[mode] = (torch.cuda.max_memory_allocated() - base) / 1e9
        release(mode)
    ops.REUSE_GRAD_PLANE = reuse

    # the gradients the modes share must agree
    backward('off')
    g_off = graphs['off'][2].grad.clone()
    backward('on')
    g_on, gx_on = graphs['on'][2].grad.clone(), graphs['on'][1].grad.clone()
    backward('forcing_only')
    gx_fo = graphs['forcing_only'][1].grad.clone()
    checks = {
        'parameter_grad_on_equals_off_bitwise': bool(torch.equal(g_on, g_off)),
        'forcing_grad_finite': bool(torch.isfinite(gx_on).all() and torch.isfinite(gx_fo).all()),
        'forcing_grad_forcing_only_vs_on_maxnorm_rel': float((gx_fo - gx_on).abs().max() / gx_on.abs().max()),
        'forcing_only_parameters_grad_is_none': graphs['forcing_only'][2].grad is None,
    }
    del g_off, g_on, gx_on, gx_fo
    for mode in MODES:
        release(mode)

    for _ in range(3):
        for mode in MODES:
            backward(mode)
            release(mode)
    k3t = {mode: [] for mode in MODES}
    step = {mode: [] for mode in MODES}
    for _ in range(args.reps):
        for mode in MODES:
            ops.PROFILE = {}
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            backward(mode)
            e1.record()
            torch.cuda.synchronize()
            release(mode)
            prof, ops.PROFILE = ops.PROFILE, None
            k3t[mode].append(sum(a.elapsed_time(b) for a, b in prof['hbv_adj_bwd']))
            step[mode].append(e0.elapsed_time(e1))

    def summary(v):
        s = sorted(v)
        return {'median': s[len(s) // 2], 'min': s[0], 'max': s[-1]}

    res = {
        'what': f'K3^T (HbvAdj adjoint, ring form) at C5: {B} basins x {T} days, nmul {NMUL}, dynamic {dyn}; '
                f'modes alternated, {args.reps} backward passes each',
        'card': card(),
        'k3t_ms': {mode: summary(k3t[mode]) for mode in MODES},
        'backward_ms': {mode: summary(step[mode]) for mode in MODES},
        'backward_peak_GB': peak,
        'parameter_plane_GB': T * B * (13 * NMUL + 2) * 4 / 1e9,
        'checks': checks,
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(json.dumps(res, indent=1) + '\n')


if __name__ == '__main__':
    main()
