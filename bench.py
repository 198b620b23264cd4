#!/usr/bin/env python
"""bench.py — basin-timesteps/sec of the HBV hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one training step of the hot path on one batch of synthetic inputs:
`Model.forward(x_dict, parameters)` (no-grad warm-up + run, nmul=16, dynamic parameters, UH
routing, BFI) followed by `streamflow.sum().backward()`.  The bench line is BASELINE.json
configs[1] ("c2": hbv, 531 basins x (365 + 730) days per GPU, dynamic [parBETA, parBETAET]).
Basins shard across GPUs with no data-path collective (weak scaling: 531 basins per GPU); the
only collective is the all-reduce of a shared-parameter gradient.

One JSON line is printed by rank 0.  `value` = device-resident throughput, `e2e` = the same
step through the public API with pinned HOST buffers (H2D of x_phy + parameters, D2H of
streamflow + loss + parameter gradient inside the timed region), `roofline` = the dominant
kernel against the measured HBM peak, `cpu_baseline` = the CPU oracle port (the reference's
PyTorch arithmetic, oracle/hbv_oracle.py) timed on this box's host cores.  `at_scale` repeats the
device-resident measurement on the north-star per-GPU shards, where the kernels are throughput-
rather than latency-bound: "shard" (same model, 22,500 basins) and "c3" (BASELINE configs[2]:
hbv_1_1p with all 14 parameters dynamic, 22,500 basins x 730 days — the HBM-bound case).

`--impl reference` times the UNMODIFIED reference (mhpi/hydrodl2's own `Hbv.forward` + autograd,
installed into the git-ignored baseline/_ref/ by scripts/install_reference.py) on the host cores,
on the SAME workload: BASELINE configs[1] in full, every step.  Only when baseline/_ref is absent
does it fall back to the oracle port (bit-exact against the reference, tests/).  `cpu_baseline`
of the B200 arm is one such step plus BASELINE configs[0] (forward only).

`--steps K` is the number of timed steps of every measurement.  `--dump-outputs DIR` writes what
the last timed step of the bench workload handed its caller to DIR/<name>.npy (float32; see
`dump_outputs`).  The inputs depend only on the arguments, so two builds run with the same
arguments can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = 'basin-timesteps/sec fwd+bwd (HBV, nmul=16)'
UNIT = 'basin-timesteps/s'
NMUL = 16
D2 = ['parBETA', 'parBETAET']
D14 = ['parBETA', 'parFC', 'parK0', 'parK1', 'parK2', 'parLP', 'parPERC', 'parUZL', 'parTT',
       'parCFMAX', 'parCFR', 'parCWH', 'parBETAET', 'parC']
WORKLOADS = {
    # BASELINE.json configs[1]: the bench line
    'c2': dict(model='hbv', cls='Hbv', dyn=D2, n_par=13, nflux=11, warm_up=365, T=730, B=531,
               label='c2: hbv fwd+bwd training step'),
    # north-star per-GPU shard (180k basins / 8 GPUs) of the same model
    'shard': dict(model='hbv', cls='Hbv', dyn=D2, n_par=13, nflux=11, warm_up=365, T=730, B=22500,
                  label='shard: hbv fwd+bwd at the north-star per-GPU basin count'),
    # BASELINE.json configs[2], one GPU's share: hbv_1_1p, all 14 parameters dynamic: HBM bound
    'c3': dict(model='hbv_1_1p', cls='Hbv_1_1p', dyn=D14, n_par=14, nflux=12, warm_up=0, T=730,
               B=22500, label='c3: hbv_1_1p fwd+bwd, all 14 parameters dynamic, 180k basins / 8 GPUs'),
}
# SURVEY.md §8 (d4) worked figures, bytes per basin-timestep (K = 32, one upstream series), quoted
# literally next to this file's own accounting (which charges the K = 1 state traffic and the
# dense gradient rows the adjoint writes): {workload: (forward, backward)}
SURVEY_BYTES = {'c2': (200.0, 292.0), 'shard': (200.0, 292.0), 'c3': (972.0, 1828.0), 'c4': (208.0, 420.0)}
SEED = 20261017
# diagnostic only: time the step without the shared-gradient all-reduce
NO_ALLREDUCE = os.environ.get('HBV_BENCH_NO_ALLREDUCE') == '1'
# capture the shared-gradient all-reduce inside the CUDA graph of the step (several GPUs)
GRAPH_ALLREDUCE = os.environ.get('HBV_BENCH_GRAPH_ALLREDUCE', '0') == '1'
# one-shot all-reduce on a parallel branch of the step's graph, one step behind (0: in line, at the
# end of the step it belongs to)
OVERLAP_ALLREDUCE = os.environ.get('HBV_BENCH_OVERLAP_ALLREDUCE', '1') == '1'


# ----------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------
def measured_peak_gbs():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


_SAMPLER_SRC = r"""
import sys, time
import pynvml as nv
nv.nvmlInit()
h = nv.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
print('max', nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM), flush=True)
while True:
    try:
        r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
    except Exception:
        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
    print(time.time(), nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), r, flush=True)
    time.sleep(0.025)
"""


class ClockSampler:
    """Samples SM clock + throttle reasons with NVML while the timed region runs.

    The sampling loop lives in a child process (a sampler thread in this process would contend
    for the GIL with the host-bound step loop and slow the very thing being timed); the parent
    only notes the wall-clock window of the timed region and filters the child's samples."""

    REASONS = {
        0x1: 'gpu_idle', 0x2: 'applications_clocks_setting', 0x4: 'sw_power_cap',
        0x8: 'hw_slowdown', 0x10: 'sync_boost', 0x20: 'sw_thermal_slowdown',
        0x40: 'hw_thermal_slowdown', 0x80: 'hw_power_brake_slowdown', 0x100: 'display_clock_setting',
    }

    def __init__(self, index: int):
        import subprocess
        self.t0 = self.t1 = None
        try:
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(vis.split(',')[index]) if vis else index
        except Exception:
            phys = index
        try:
            self.proc = subprocess.Popen([sys.executable, '-c', _SAMPLER_SRC, str(phys)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def start(self):
        self.t0 = time.time()

    def stop(self):
        # the child is ended right here: NVML queries serialise with kernel launches in the
        # driver, so a sampler left running would slow every later measurement of this process
        self.t1 = time.time()
        self.out = ''
        if self.proc is not None:
            time.sleep(0.03)
            self.proc.terminate()
            try:
                self.out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
            self.proc = None
            self.ran = True

    def summary(self):
        if not getattr(self, 'ran', False):
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvml unavailable']}
        out = self.out
        max_mhz, inside, all_s, reasons = None, [], [], set()
        for ln in out.splitlines():
            f = ln.split()
            try:
                if f[0] == 'max':
                    max_mhz = int(f[1])
                    continue
                ts, mhz, r = float(f[0]), int(f[1]), int(f[2])
            except Exception:
                continue
            all_s.append((ts, mhz))
            if self.t0 is not None and self.t0 <= ts <= self.t1:
                inside.append(mhz)
                for bit, name in self.REASONS.items():
                    if r & bit and name != 'gpu_idle':
                        reasons.add(name)
        if not inside and all_s and self.t0 is not None:
            # timed region shorter than one sampling period: take the nearest sample
            mid = 0.5 * (self.t0 + self.t1)
            inside = [min(all_s, key=lambda s: abs(s[0] - mid))[1]]
        if not inside:
            return {'sm_mhz': None, 'sm_max_mhz': max_mhz, 'reasons': ['nvml unavailable']}
        return {'sm_mhz': statistics.median(inside), 'sm_max_mhz': max_mhz,
                'reasons': sorted(reasons), 'samples': len(inside)}


def synthetic_forcing(T, B, seed):
    """[T, B, 3] = (prcp, tmean, pet) on the CPU (SURVEY.md §8 d2): seasonal temperature crossing
    the snow threshold, 50 % dry days, seasonal PET.  (bench.py's own generator: the B200 arm does
    not import anything from oracle/.)"""
    g = torch.Generator().manual_seed(seed)
    d = torch.arange(T, dtype=torch.float32).view(T, 1)
    ob = torch.rand(1, B, generator=g) * 16 - 8
    season = torch.sin(2 * math.pi * (d - 110) / 365)
    tmean = 5 + 12 * season + ob + 4 * torch.randn(T, B, generator=g)
    prcp = 5 * torch.relu(torch.randn(T, B, generator=g))
    pet = torch.relu(2 + 2 * season) + 0.5 * torch.rand(T, B, generator=g)
    return torch.stack([prcp, tmean, pet], dim=-1).contiguous()


def make_inputs(wl, B, seed, device=None, pin=False):
    """Synthetic forcings (SURVEY.md §8 d2) + raw parameters ~ N(0,1)."""
    T = wl['warm_up'] + wl['T']
    ncol = wl['n_par'] * NMUL + 2
    if device is not None and B > 4096:
        # large shard: generate on the device (same distributions, different stream)
        g = torch.Generator(device=device).manual_seed(seed)
        d = torch.arange(T, dtype=torch.float32, device=device).view(T, 1)
        ob = torch.rand(1, B, generator=g, device=device) * 16 - 8
        season = torch.sin(2 * math.pi * (d - 110) / 365)
        tmean = 5 + 12 * season + ob + 4 * torch.randn(T, B, generator=g, device=device)
        prcp = 5 * torch.relu(torch.randn(T, B, generator=g, device=device))
        pet = torch.relu(2 + 2 * season) + 0.5 * torch.rand(T, B, generator=g, device=device)
        x = torch.stack([prcp, tmean, pet], dim=-1).contiguous()
        del tmean, prcp, pet
        p = torch.empty(T, B, ncol, device=device)
        tb = max(1, T // 8)
        for t0 in range(0, T, tb):      # in slabs: randn needs no second full-size temporary
            p[t0:t0 + tb].normal_(generator=g)
        return x, p
    x = synthetic_forcing(T, B, seed=seed)
    p = torch.randn(T, B, ncol, generator=torch.Generator().manual_seed(seed + 1))
    if pin:
        x, p = x.pin_memory(), p.pin_memory()
    return x, p


def model_config(wl):
    return {'warm_up': wl['warm_up'], 'dynamic_params': {wl['cls']: wl['dyn']}, 'nmul': NMUL}


DUMP_LIMIT = 64 * 10 ** 6     # bytes written by --dump-outputs, .npy headers included
NPY_HEADER = 128


def dump_outputs(dirname, out, loss, grad, shared_grad=None):
    """Write one training step's results as float32 `dirname/<name>.npy`: every series of `out`
    (`Model.forward`'s dict), `loss`, `grad_parameters` (the gradient w.r.t. `parameters`) and, if
    given, `grad_shared` (the all-reduced shared-bias gradient).  When the full arrays exceed
    DUMP_LIMIT, every per-basin array keeps the same seeded subset of basins, in ascending order."""
    import numpy as np
    B = grad.shape[1]
    arrays = {k: (v, 0 if v.dim() == 1 else 1) for k, v in out.items() if v is not None}
    arrays.update(loss=(loss, None), grad_parameters=(grad, 1))
    if shared_grad is not None:
        arrays['grad_shared'] = (shared_grad, None)
    for k, (v, ax) in arrays.items():
        assert ax is None or v.shape[ax] == B, f'{k}: {tuple(v.shape)} has no basin axis of size {B}'
    room = DUMP_LIMIT - NPY_HEADER * len(arrays) - sum(4 * v.numel() for v, ax in arrays.values() if ax is None)
    per_basin = sum(4 * v.numel() // B for v, ax in arrays.values() if ax is not None)
    keep = min(B, room // per_basin)
    idx = None
    if keep < B:
        idx = torch.randperm(B, generator=torch.Generator().manual_seed(SEED))[:keep].sort().values
    os.makedirs(dirname, exist_ok=True)
    for k, (v, ax) in arrays.items():
        v = v.detach()
        if idx is not None and ax is not None:
            v = v.index_select(ax, idx.to(v.device))
        np.save(os.path.join(dirname, k + '.npy'), v.float().cpu().numpy())


# algorithmic bytes per basin-timestep (DESIGN.md §4; SURVEY.md §8 d4), nmul = 16:
# every contract input read once, every output written once
def bytes_fwd(wl, K=16):
    # forcings + dynamic parameters read, flux planes written, state checkpoint every K steps
    return 4 * (3 + len(wl['dyn']) * NMUL + wl['nflux']) + 5 * NMUL * 4 / K


def bytes_bwd(wl, K=16, n_g=1, fused=False):
    # forcings + dynamic parameters + n_g upstream series + stored states read; gradient written:
    # the dynamic columns only when the caller pre-zeroed the dense plane (memset), the whole dense
    # [B, ncol] row — a contract output, zeros included — when the adjoint writes it itself
    ncol = wl['n_par'] * NMUL + 2
    n_dyn = len(wl['dyn']) * NMUL
    written = ncol if fused else n_dyn
    return 4 * (3 + n_dyn + n_g + written) + 5 * NMUL * 4 / K


def per_unit_bytes(wl, K, fused=False):
    return {'hbv_bwd': bytes_bwd(wl, K, fused=fused), 'hbv_fwd': bytes_fwd(wl, K), 'hbv_fwd_warmup': 12.0,
            'route_fwd': 32.0,    # 4 series read + 4 routed series written
            'route_bwd': 12.0}    # streamflow-only loss: read g, read x, write g_in (1 series)


def config_of(wl, B, world):
    """The `config` object both arms print (identical for the same workload and GPU count)."""
    ncol = wl['n_par'] * NMUL + 2
    return {
        'workload': describe(wl, B),
        'basins_per_gpu': B, 'basins_total': B * world, 'warm_up': wl['warm_up'],
        'steps_counted': wl['T'], 'nmul': NMUL, 'dynamic_params': list(wl['dyn']),
        'parallelism': f'basin-sharded x{world}, all-reduce of the shared-bias gradient only',
        'l2': 'inputs larger than L2: parameters + gradient = '
              f'{2 * (wl["warm_up"] + wl["T"]) * B * ncol * 4 / 1e6:.0f} MB per step vs 126 MB L2',
    }


def describe(wl, B):
    return (f"{wl['label']}, {B} basins/GPU x ({wl['warm_up']} warm-up + {wl['T']}) days, nmul {NMUL}, "
            f"{len(wl['dyn'])} dynamic parameters {wl['dyn'] if len(wl['dyn']) <= 3 else '(all)'}, "
            f"UH routing + BFI, loss = streamflow.sum()")


# ----------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the unmodified reference (baseline/_ref) on the host cores,
# else the oracle port
# ----------------------------------------------------------------------------------------------
REF_DIR = os.path.join(ROOT, 'baseline', '_ref')


def load_reference():
    """The unmodified reference package from baseline/_ref (scripts/install_reference.py), or None."""
    if not os.path.isdir(os.path.join(REF_DIR, 'hydrodl2')):
        return None
    os.environ.setdefault('CI', '1')          # licence prompt bypass (hydrodl2/__init__.py:103-122)
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    try:
        import logging
        logging.getLogger('hydrodl2').setLevel(logging.ERROR)
        import hydrodl2 as ref
        return ref
    except Exception as exc:    # pragma: no cover
        print(f'bench.py: baseline/_ref present but not importable ({exc}); using the oracle port', file=sys.stderr)
        return None


class CpuArm:
    """One workload on the host: the reference's own module (kind 'reference') or the oracle port."""

    def __init__(self, wl):
        self.wl = wl
        self.ref = load_reference()
        self.kind = 'reference' if self.ref is not None else 'port'
        self.model = None
        if self.ref is not None:
            M = self.ref.load_model(wl['model'], ver_name=wl['cls'])
            self.model = M(model_config(wl), device=torch.device('cpu'))

    def train_step(self, x, p):
        """fwd + bwd of the whole workload (warm-up + run); -> seconds."""
        wl = self.wl
        pr = p.detach().clone().requires_grad_(True)
        t0 = time.perf_counter()
        if self.model is not None:
            out = self.model({'x_phy': x}, pr)
        else:
            from oracle import hbv_oracle as O
            out, _ = O.forward_packed(wl['model'], x, pr, nmul=NMUL, warm_up=wl['warm_up'], dynamic_params=wl['dyn'])
        out['streamflow'].sum().backward()
        dt = time.perf_counter() - t0
        self.last = (out, pr.grad)
        return dt

    def forward_only(self, x, p):
        """BASELINE configs[0]: forward under no_grad over the run rows only (no warm-up); -> seconds."""
        wl = self.wl
        W = wl['warm_up']
        xs, ps = x[W:].contiguous(), p[W:].contiguous()
        t0 = time.perf_counter()
        with torch.no_grad():
            if self.ref is not None:
                M = self.ref.load_model(wl['model'], ver_name=wl['cls'])
                m0 = M(dict(model_config(wl), warm_up=0), device=torch.device('cpu'))
                m0({'x_phy': xs}, ps)
            else:
                from oracle import hbv_oracle as O
                O.forward_packed(wl['model'], xs, ps, nmul=NMUL, warm_up=0, dynamic_params=wl['dyn'])
        return time.perf_counter() - t0


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    wl = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    B = wl['B'] if args.basins is None else args.basins
    if B > 531:
        print('bench.py --impl reference: the CPU arm runs the bench workload (c2) only', file=sys.stderr)
    x, p = make_inputs(wl, B, SEED)
    arm = CpuArm(wl)
    for _ in range(args.warmup):
        arm.train_step(x, p)
    tot = 0.0
    for _ in range(args.steps):
        tot += arm.train_step(x, p)
    if args.dump_outputs:
        out, grad = arm.last
        dump_outputs(args.dump_outputs, out, out['streamflow'].sum(), grad)
    val = args.steps * B * wl['T'] / tot
    what = ("unmodified mhpi/hydrodl2 (baseline/_ref): Hbv.forward + autograd" if arm.kind == 'reference'
            else 'oracle port of the reference (oracle/hbv_oracle.py; baseline/_ref absent)')
    sample = (f'{what}; every step = the full workload, {B} basins x ({wl["warm_up"]} warm-up + {wl["T"]}) days, '
              f'fwd+bwd, {cores} threads')
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * tot / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': config_of(wl, B, max(1, args.gpus)),
        'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': cores, 'kind': arm.kind, 'sample': sample},
        'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(line)
    return 0


# ----------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------
def run_b200(args):
    from hydrodl2_b200 import _cabi, dist as D, ops
    import hydrodl2_b200 as hydrodl2

    if not torch.cuda.is_available():
        print('bench.py: no CUDA device — the B200 arm has no CPU fallback', file=sys.stderr)
        return 2
    # keep stdout to the one JSON line: NCCL prints its version banner there at VERSION / WARN level
    if os.environ.get('NCCL_DEBUG', '').upper() in ('VERSION', 'WARN'):
        os.environ.pop('NCCL_DEBUG')
    rank, local, world = D.init_from_env()
    if world != args.gpus and rank == 0:
        print(f'bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; using {world}', file=sys.stderr)
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    numa = 'unchanged (HBV_BENCH_NO_NUMA=1)' if os.environ.get('HBV_BENCH_NO_NUMA') == '1' else D.bind_to_gpu_numa_node(local)
    _cabi.load()
    peak, peak_src = measured_peak_gbs()
    # the shared-gradient all-reduce: the library's one-shot kernel over NVLink peer memory
    # (csrc/allreduce.cu) when symmetric memory can be set up, else NCCL; HBV_BENCH_ONESHOT=0 keeps NCCL
    oneshot = False
    if world > 1 and os.environ.get('HBV_BENCH_ONESHOT', '1') != '0':
        oneshot = all([D.enable_oneshot_allreduce(w['n_par'] * NMUL + 2, dev)
                       for w in ({'n_par': 13}, {'n_par': 14})])

    def build(wl, B, pin):
        Model = hydrodl2.load_model(wl['model'], ver_name=wl['cls'])
        x, p = make_inputs(wl, B, SEED + rank, device=dev, pin=pin)
        model = Model(dict(model_config(wl), ckpt_interval=args.ckpt), device=dev)
        return model, x, p

    def k_eff(wl, B):      # the checkpoint interval the run actually uses (0 = library default)
        if args.ckpt:
            return args.ckpt
        Model = hydrodl2.load_model(wl['model'], ver_name=wl['cls'])
        spec = Model(model_config(wl), device=dev)._spec(wl['dyn'], True)
        ncol = wl['n_par'] * NMUL + 2
        import ctypes
        return int(_cabi.load().hbv_b200_auto_ckpt_desc(ctypes.byref(ops.make_desc(spec, wl['T'], B, 3, ncol, 0))))

    def train_step(model, x_dev, p_dev, allreduce=True):
        p_dev.grad = None
        out = model({'x_phy': x_dev}, p_dev)
        loss = out['streamflow'].sum()
        loss.backward()
        # gradient of a bias on the static-parameter row shared by all basins (stands in for
        # the shared NN weights): the one quantity that needs a cross-GPU reduction
        gshared = p_dev.grad[-1].sum(dim=0)
        if allreduce and not NO_ALLREDUCE:
            D.allreduce_shared_grad(gshared)
        return out, loss, gshared

    def fwd_only(model, x, p):
        with torch.no_grad():
            return model({'x_phy': x}, p)

    def timed(fn, steps, warmup, sampler=None, tail=None):
        # tail: work that closes the K steps and belongs to them (the flush of a pipelined reduction)
        for _ in range(warmup):
            fn()
        if tail:
            tail()
        torch.cuda.synchronize(dev)
        D.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if sampler:
            sampler.start()
        e0.record()
        for _ in range(steps):
            fn()
        if tail:
            tail()
        e1.record()
        torch.cuda.synchronize(dev)
        if sampler:
            sampler.stop()
        D.barrier()
        return D.max_over_ranks(e0.elapsed_time(e1), dev)   # ms, max over ranks

    def timed_with_kernels(fn, steps, warmup, sampler=None):
        """-> (ms per step, {kernel group: mean ms per call over the timed steps})."""
        ops.PROFILE = {}
        ms = timed(fn, steps, warmup, sampler) / steps
        prof, ops.PROFILE = ops.PROFILE, None
        torch.cuda.synchronize(dev)
        kms = {}
        for name, evs in prof.items():
            per_step = len(evs) // (steps + warmup)
            evs = evs[warmup * per_step:]
            kms[name] = sum(a.elapsed_time(b) for a, b in evs) / max(1, len(evs))
        return ms, kms

    def fused_fill(wl, B):     # does the adjoint write the dense gradient rows itself? (ops.py policy)
        Model = hydrodl2.load_model(wl['model'], ver_name=wl['cls'])
        spec = Model(model_config(wl), device=dev)._spec(wl['dyn'], True)
        return bool(ops._fused_zero_fill(spec, wl['n_par'] * NMUL + 2, B))

    def rows_written(wl, B):   # ... in the timed steps: not when a clean plane is kept between them
        return fused_fill(wl, B) and not ops.REUSE_GRAD_PLANE

    def roofline_of(wl, B, kms, kernel, traffic_key=None):
        units = B * (wl['T'] if kernel != 'hbv_fwd_warmup' else wl['warm_up'])
        per_unit = per_unit_bytes(wl, k_eff(wl, B), rows_written(wl, B))[kernel]
        achieved = per_unit * units / (kms[kernel] * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, 'profiles', 'roofline_traffic.json')
        if traffic_key and os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get(traffic_key, {}).get(kernel)
            except Exception:
                traffic = None
        r = {'bound': 'hbm', 'kernel': kernel, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
             'frac': achieved / peak, 'traffic': traffic, 'peak_source': peak_src,
             'gradient_plane': ('dense rows written by the adjoint' if rows_written(wl, B) else
                                'zero background (a clean plane kept between steps, else a memset / the adjoint\'s own zero fill) + dynamic columns'),
             'algorithmic_bytes_per_basin_step': per_unit, 'kernel_ms': kms[kernel]}
        sb = SURVEY_BYTES.get(traffic_key)
        if sb and kernel in ('hbv_fwd', 'hbv_bwd'):
            # SURVEY.md §8 (d4) literal figure (no K = 1 state traffic, gradient = dynamic columns only)
            lit = sb[0] if kernel == 'hbv_fwd' else sb[1]
            r['algorithmic_bytes_survey'] = lit
            r['frac_survey'] = lit * units / (kms[kernel] * 1e-3) / 1e9 / peak
        return r

    # ---------------- the bench workload: device-resident throughput + per-kernel roofline -----
    wl = WORKLOADS[args.workload]
    B = wl['B'] if args.basins is None else args.basins
    T_MAIN = wl['T']
    model, x_host, p_host = build(wl, B, pin=True)
    x_dev = x_host.to(dev)
    p_dev = p_host.to(dev).requires_grad_(True)
    n0 = _cabi.launch_count()
    train_step(model, x_dev, p_dev)
    torch.cuda.synchronize(dev)
    launches_per_step = _cabi.launch_count() - n0

    sampler = ClockSampler(local)     # child process; up and sampling well before the timed region
    # per-kernel device times (eager, CUDA events around every C-ABI call)
    ms_eager, kms = timed_with_kernels(lambda: train_step(model, x_dev, p_dev), args.steps, args.warmup)
    # the timed step: eager by default; --graph replays the same step from a CUDA graph
    graph_note = 'eager'
    step_fn = lambda: train_step(model, x_dev, p_dev)   # noqa: E731
    step_tail = None
    if args.graph:
        try:
            from hydrodl2_b200.graphs import GraphedStep
            if world == 1:
                gstep = GraphedStep(lambda: train_step(model, x_dev, p_dev, allreduce=False), warmup=3, device=dev)
                step_fn = gstep.replay
                graph_note = 'cuda graph replay of the whole step (hydrodl2_b200.graphs.GraphedStep)'
            elif oneshot and not NO_ALLREDUCE and OVERLAP_ALLREDUCE:
                # The collective is a plain kernel of this library, captured with the step — on a
                # parallel branch of the graph: replay i reduces the shared gradient of step i-1
                # (staged by replay i-1) while it computes step i, so the cross-rank wait of the
                # reduction is off the step's critical path (rank skew up to one step is absorbed).
                # Every step's gradient is still reduced, one step late; the last one by `tail`,
                # inside the timed region.
                n_sh = wl['n_par'] * NMUL + 2
                stage = torch.zeros(n_sh, device=dev)        # step i-1's local shared gradient
                reduced = torch.zeros(n_sh, device=dev)      # the latest finished reduction
                comm = torch.cuda.Stream(dev)

                def overlapped_step():
                    cur = torch.cuda.current_stream(dev)
                    comm.wait_stream(cur)
                    with torch.cuda.stream(comm):
                        reduced.copy_(stage)
                        D.allreduce_shared_grad(reduced)
                    out, loss, gsh = train_step(model, x_dev, p_dev, allreduce=False)
                    cur.wait_stream(comm)
                    stage.copy_(gsh)
                    return out, loss, reduced

                def flush_reduction():
                    reduced.copy_(stage)
                    D.allreduce_shared_grad(reduced)

                gstep = GraphedStep(overlapped_step, warmup=3, device=dev)
                step_fn, step_tail = gstep.replay, flush_reduction
                graph_note = ('cuda graph replay of the whole step; the one-shot all-reduce of the shared gradient '
                              '(csrc/allreduce.cu, NVLink peer memory) runs on a parallel branch of the graph, one '
                              'step behind: replay i reduces step i-1\'s gradient while computing step i, the '
                              'last one is flushed inside the timed region')
            elif oneshot and not NO_ALLREDUCE:
                # the collective is a plain kernel of this library: captured with the step
                gstep = GraphedStep(lambda: train_step(model, x_dev, p_dev, allreduce=True), warmup=3, device=dev)
                step_fn = gstep.replay
                graph_note = ('cuda graph replay of the whole step incl. the one-shot all-reduce of the shared '
                              'gradient over NVLink peer memory (csrc/allreduce.cu)')
            elif GRAPH_ALLREDUCE and not NO_ALLREDUCE:
                # the shared-gradient all-reduce is captured with the step (thread-local capture mode:
                # NCCL's watchdog thread may issue CUDA calls while this thread captures)
                gstep = GraphedStep(lambda: train_step(model, x_dev, p_dev, allreduce=True), warmup=3, device=dev,
                                    capture_error_mode='thread_local')
                step_fn = gstep.replay
                graph_note = ('cuda graph replay of the whole step incl. the NCCL all-reduce of the shared '
                              'gradient (hydrodl2_b200.graphs.GraphedStep)')
            else:
                # each rank replays its own step, then the shared-gradient all-reduce runs eagerly on
                # the graph's static output
                gstep = GraphedStep(lambda: train_step(model, x_dev, p_dev, allreduce=False), warmup=3, device=dev)

                def step_fn():
                    res = gstep.replay()
                    if not NO_ALLREDUCE:
                        D.allreduce_shared_grad(res[2])
                    return res
                graph_note = ('cuda graph replay of the step (hydrodl2_b200.graphs.GraphedStep) + eager NCCL '
                              'all-reduce of the shared gradient')
        except Exception as exc:   # pragma: no cover - depends on driver / NCCL
            graph_note = f'eager (graph capture failed: {type(exc).__name__}: {exc})'
            step_fn = lambda: train_step(model, x_dev, p_dev)   # noqa: E731
            step_tail = None
            torch.cuda.synchronize(dev)
    last = []
    timed_fn = step_fn
    if args.dump_outputs:
        def timed_fn():
            last[:] = [step_fn()]
    ms_step = timed(timed_fn, args.steps, args.warmup, sampler, tail=step_tail) / args.steps
    if args.dump_outputs and rank == 0:
        out, loss, gshared = last[0]
        dump_outputs(args.dump_outputs, out, loss, p_dev.grad, gshared)
    value = world * B * T_MAIN / (ms_step * 1e-3)
    # The same step with a freshly zeroed dense gradient plane at every step (the clean-plane cache
    # of ops.py switched off): what the 488 MB memset costs.  In the timed loop above the plane of
    # the previous step is handed out again without it — nobody references it any more and nobody
    # modified it in place, and the adjoint rewrites every entry that can be non-zero.
    ms_memset = None
    plane_cached = bool(ops.REUSE_GRAD_PLANE)
    if plane_cached and world == 1:
        ops.REUSE_GRAD_PLANE = False
        try:
            fn2 = lambda: train_step(model, x_dev, p_dev, allreduce=False)   # noqa: E731
            if args.graph:
                from hydrodl2_b200.graphs import GraphedStep
                fn2 = GraphedStep(fn2, warmup=3, device=dev).replay
            ms_memset = timed(fn2, args.steps, args.warmup) / args.steps
        finally:
            ops.REUSE_GRAD_PLANE = True
    dom = max(kms, key=kms.get)
    roofline = roofline_of(wl, B, kms, dom, traffic_key=args.workload)
    if B * NMUL < 148 * 2048 // 4:
        roofline['note'] = (f'{B} basins x 16 = {B * NMUL} lanes (<{100 * B * NMUL / (148 * 2048):.0f}% of '
                            'one B200 wave): the step is latency-bound, see at_scale for the '
                            'throughput regime')

    ms_fwd, kms_fwd = timed_with_kernels(lambda: fwd_only(model, x_dev, p_dev), args.steps, args.warmup)
    fwd = {'value': world * B * T_MAIN / (ms_fwd * 1e-3), 'unit': UNIT, 'ms_per_step': ms_fwd,
           'kernel_ms': kms_fwd}

    # ---------------- end to end with host buffers ----------------
    e2e = None
    if not x_host.is_cuda:   # shard-sized inputs are generated on the device: no host copy to time
        e2e = _e2e(args, dev, world, wl, B, model, x_host, p_host, x_dev, p_dev, train_step, timed)
    del x_dev, p_dev, x_host, p_host, model
    ops.release_grad_planes()      # (idle cached gradient planes of the finished workload)
    torch.cuda.empty_cache()

    # ---------------- north-star per-GPU shards ----------------
    at_scale = None
    if not args.no_at_scale and args.workload == 'c2' and args.basins is None:
        at_scale = {}
        for name in ('shard', 'c3'):
            w2 = WORKLOADS[name]
            Bs = w2['B']
            model_s, xs, ps = build(w2, Bs, pin=False)
            ps.requires_grad_(True)
            s_steps, s_warm = args.steps, 3
            ms_s, kms_s = timed_with_kernels(lambda: train_step(model_s, xs, ps), s_steps, s_warm)
            ms_sf, kms_sf = timed_with_kernels(lambda: fwd_only(model_s, xs, ps), s_steps, s_warm)
            ms_s_fill = None          # the same step with the dense plane (re)written at every step
            if ops.REUSE_GRAD_PLANE:
                ops.REUSE_GRAD_PLANE = False
                try:
                    ps.grad = None
                    ops.release_grad_planes()
                    ms_s_fill = timed(lambda: train_step(model_s, xs, ps), s_steps, s_warm) / s_steps
                finally:
                    ops.REUSE_GRAD_PLANE = True
            at_scale[name] = {
                'workload': describe(w2, Bs),
                'value': world * Bs * w2['T'] / (ms_s * 1e-3), 'unit': UNIT, 'ms_per_step': ms_s,
                'ms_per_step_plane_rewritten_every_step': ms_s_fill,
                'fwd_value': world * Bs * w2['T'] / (ms_sf * 1e-3), 'fwd_ms_per_step': ms_sf,
                'kernel_ms': kms_s, 'fwd_kernel_ms': kms_sf,
                'roofline': roofline_of(w2, Bs, kms_s, 'hbv_bwd', traffic_key=name),
                'roofline_fwd': roofline_of(w2, Bs, kms_s, 'hbv_fwd', traffic_key=name),
            }
            del model_s, xs, ps
            ops.release_grad_planes()      # (idle cached gradient planes of the finished workload)
            torch.cuda.empty_cache()

    # BASELINE configs[3] and [4] at their per-GPU sizes (scripts/bench_configs.py): c4 = hbv_2_hourly,
    # 2,500 units per GPU x 17,520 hourly steps (weak: 20k units on 8 GPUs); c5 = hbv_adj, 10,000 basins
    # in total, i.e. 10,000 / N per GPU (strong).  Same timing rules (CUDA events, max over ranks).
    if at_scale is not None and not args.no_configs:
        import importlib.util
        spec_ = importlib.util.spec_from_file_location('bench_configs', os.path.join(ROOT, 'scripts', 'bench_configs.py'))
        cfgs = importlib.util.module_from_spec(spec_)
        spec_.loader.exec_module(cfgs)
        for name, fn, kw in (('c4', cfgs.run_c4, {'B': 2500}), ('c5', cfgs.run_c5, {'B': max(1, 10000 // world)})):
            try:
                res = fn(args.steps, dev=dev, seed_offset=rank, **kw)
            except Exception as exc:      # pragma: no cover - keep the bench line alive
                at_scale[name] = {'error': f'{type(exc).__name__}: {exc}'}
                ops.release_grad_planes()      # (idle cached gradient planes of the finished workload)
                torch.cuda.empty_cache()
                continue
            ms_max = D.max_over_ranks(res['ms_per_step'], dev)
            msf_max = D.max_over_ranks(res['fwd_ms_per_step'], dev)
            units = res['units_per_gpu'] * world
            entry = {'workload': res['config'], 'value': units / (ms_max * 1e-3), 'unit': UNIT, 'ms_per_step': ms_max,
                     'fwd_value': units / (msf_max * 1e-3), 'fwd_ms_per_step': msf_max,
                     'kernel_ms': res['kernel_ms'], 'checks': res['checks'],
                     'scaling': 'weak' if name == 'c4' else 'strong (10,000 basins in total)'}
            for leg, kern in (('roofline', res['bwd_kernel']), ('roofline_fwd', res['fwd_kernel'])):
                by = res['bytes'][kern]
                ach = by['ours'] * res['units_per_gpu'] / (res['kernel_ms'][kern] * 1e-3) / 1e9
                entry[leg] = {'bound': 'hbm', 'kernel': kern, 'achieved': ach, 'peak': peak, 'unit': 'GB/s',
                              'frac': ach / peak, 'traffic': None, 'peak_source': peak_src,
                              'algorithmic_bytes_per_basin_step': by['ours'], 'kernel_ms': res['kernel_ms'][kern]}
                if by.get('survey'):
                    entry[leg]['algorithmic_bytes_survey'] = by['survey']
                    entry[leg]['frac_survey'] = by['survey'] * res['units_per_gpu'] / (res['kernel_ms'][kern] * 1e-3) / 1e9 / peak
            at_scale[name] = entry
            ops.release_grad_planes()      # (idle cached gradient planes of the finished workload)
            torch.cuda.empty_cache()

    # ---------------- CPU baseline (rank 0, N = 1 only) ----------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        wl_c = WORKLOADS['c2']          # the CPU leg always runs the bench workload at its full size
        xc, pc_ = make_inputs(wl_c, wl_c['B'], SEED)
        arm = CpuArm(wl_c)
        dt = arm.train_step(xc, pc_)
        dt_f = min(arm.forward_only(xc, pc_) for _ in range(2))
        what = ('unmodified mhpi/hydrodl2 (baseline/_ref)' if arm.kind == 'reference'
                else 'oracle port of the reference (baseline/_ref absent)')
        cpu_baseline = {
            'value': wl_c['B'] * wl_c['T'] / dt, 'unit': UNIT, 'cores': cores, 'kind': arm.kind,
            'sample': f"{what}: BASELINE configs[1] in full, {wl_c['B']} basins x ({wl_c['warm_up']} warm-up + "
                      f"{wl_c['T']}) days, fwd+bwd, one step, {dt:.1f} s of CPU work",
            'c1_fwd': {'value': wl_c['B'] * wl_c['T'] / dt_f, 'unit': UNIT, 'seconds': dt_f,
                       'sample': f"BASELINE configs[0]: hbv forward (no_grad), {wl_c['B']} basins x {wl_c['T']} days, "
                                 f"nmul {NMUL}, best of 2"},
        }
        if not args.no_cpu_slices:
            # BASELINE configs 3-5 on bounded slices (SURVEY §8 d5; reference cost is linear in basins)
            try:
                import importlib.util
                sp = importlib.util.spec_from_file_location('cpu_slices', os.path.join(ROOT, 'scripts', 'cpu_slices.py'))
                cs = importlib.util.module_from_spec(sp)
                sp.loader.exec_module(cs)
                cpu_baseline['slices'] = cs.run(nb=128, nb_hourly=32, nb_adj=16)
            except Exception as exc:     # pragma: no cover
                cpu_baseline['slices'] = {'error': f'{type(exc).__name__}: {exc}'}

    if rank == 0:
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_step, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': config_of(wl, B, world),
            'run_info': {'ckpt_interval': k_eff(wl, B), 'launch': graph_note, 'eager_ms_per_step': ms_eager,
                         'gradient_plane': ('clean plane kept between steps (released + unmodified => no memset / no '
                                            'zero fill by the adjoint; hydrodl2_b200.ops._clean_plane)' if plane_cached else
                                            ('zeroed by the adjoint itself' if fused_fill(wl, B) else 'memset every step')),
                         'ms_per_step_plane_memset_every_step': ms_memset,
                         'shared_grad_allreduce': (('one-shot kernel over NVLink peer memory'
                                                    + (', overlapped with the next step (one step behind)'
                                                       if step_tail is not None else '')) if oneshot else
                                                   ('nccl' if world > 1 else 'none (one GPU)')),
                         'host_affinity': numa},
            'clocks': sampler.summary(), 'e2e': e2e, 'gpu_launches': launches_per_step * args.steps,
            'gpu_launches_per_step': launches_per_step,
            'roofline': roofline, 'cpu_baseline': cpu_baseline, 'fwd': fwd, 'kernel_ms': kms,
            'at_scale': at_scale,
        }
        emit(line)
    if world > 1:
        import torch.distributed as dist
        if oneshot and any(o is not None and o.timed_out() for o in D._ONESHOT.values()):
            print('bench.py: the one-shot all-reduce timed out waiting for a peer — results invalid', file=sys.stderr)
            return 3
        dist.destroy_process_group()
    return 0


def _e2e(args, dev, world, wl, B, model, x_host, p_host, x_dev, p_dev, train_step, timed):
    """Same step through the public API with pinned HOST buffers, every copy inside the timed
    region.  Two loops are timed: `serial` (upload, step, download, wait — one after the other) and
    the reported one, `hydrodl2_b200.hostio.PipelinedSteps` (double-buffered inputs on three
    streams, so a step's upload and the previous step's download overlap the kernels; every step
    still moves its own inputs and results)."""
    from hydrodl2_b200.hostio import PipelinedSteps
    g_host = torch.empty_like(p_host).pin_memory()
    q_host = torch.empty(wl['T'], B, 1).pin_memory()
    l_host = torch.empty(()).pin_memory()
    xd = torch.empty_like(x_dev)
    pd = torch.empty_like(p_dev.detach()).requires_grad_(True)

    def e2e_step():
        xd.copy_(x_host, non_blocking=True)
        with torch.no_grad():
            pd.copy_(p_host, non_blocking=True)
        out, loss, _ = train_step(model, xd, pd)
        q_host.copy_(out['streamflow'], non_blocking=True)
        l_host.copy_(loss.detach(), non_blocking=True)
        g_host.copy_(pd.grad, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()   # the caller needs the results on the host

    e2e_steps = args.steps
    ms_serial = timed(e2e_step, e2e_steps, 3) / e2e_steps
    del xd, pd, g_host, q_host, l_host

    def pipe_step(inp):
        out, loss, _ = train_step(model, inp['x_phy'], inp['parameters'])
        return {'streamflow': out['streamflow'], 'loss': loss, 'grad': inp['parameters'].grad}

    # column-sparse staging: upload only what the kernels read of `parameters` (the dynamic blocks +
    # the last row + the last warm-up row), download only the non-zero part of its gradient into a
    # pinned host plane zeroed once — the host still holds the full dense gradient (hostio.py)
    host_in = {'x_phy': x_host, 'parameters': p_host}
    fp = model.io_footprint(p_host.shape[0])
    pipe = PipelinedSteps(pipe_step, host_in, dev, leaf_names=('parameters',),
                          in_footprints={'parameters': fp['read']}, out_footprints={'grad': fp['grad']})

    def pipe_run(n):
        for _ in range(n):
            pipe.step(host_in)
        pipe.drain()      # every upload, kernel and download of the n steps has completed

    pipe_run(3)
    torch.cuda.synchronize(dev)
    from hydrodl2_b200 import dist as D
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pipe_run(e2e_steps)
    e1.record()
    torch.cuda.synchronize(dev)
    D.barrier()
    ms_e2e = D.max_over_ranks(e0.elapsed_time(e1), dev) / e2e_steps
    h2d, d2h = int(pipe.h2d_bytes), int(pipe.d2h_bytes)       # counted from the copies the loop issued
    # the downloaded host plane is the dense gradient: check it against the device tensor once
    hb = pipe.step(host_in)
    pipe.drain()
    p_chk = p_host.to(dev).requires_grad_(True)
    train_step(model, x_host.to(dev), p_chk)
    torch.cuda.synchronize(dev)
    dense_ok = bool(torch.equal(hb['grad'], p_chk.grad.cpu()))
    del p_chk
    return {'value': world * B * wl['T'] / (ms_e2e * 1e-3), 'unit': UNIT, 'ms_per_step': ms_e2e,
            'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
            'dense_bytes_per_step': {'h2d': x_host.numel() * 4 + p_host.numel() * 4,
                                     'd2h': p_host.numel() * 4 + wl['T'] * B * 4 + 4},
            'host_gradient_equals_dense_device_gradient': dense_ok,
            'serial_ms_per_step': ms_serial,
            'pcie_GBps': {'h2d': h2d / (ms_e2e * 1e-3) / 1e9, 'd2h': d2h / (ms_e2e * 1e-3) / 1e9},
            # how the column blocks crossed PCIe on THIS host (hostio.pick_block_copy times both ways
            # on the first step: copy engine 2-D copies vs the GPU reading / writing pinned memory)
            'block_copy': {f'{d}:{n}': m for (d, n), m in pipe.block_copy.items()},
            'what': 'pinned host x_phy + parameters -> device, Model.forward + backward, '
                    'streamflow + loss + parameter gradient -> pinned host; double-buffered on '
                    'upload / compute / download streams (hydrodl2_b200.hostio.PipelinedSteps), '
                    'each step moves its own inputs and results; column-sparse: of `parameters` only '
                    'the entries the kernels read (dynamic blocks, last row, last warm-up row) go up, '
                    'of its gradient only the non-zero entries come down, into a pinned host plane '
                    'zeroed once (the host holds the full dense gradient: '
                    'host_gradient_equals_dense_device_gradient); serial_ms_per_step = whole-tensor '
                    'copies, no overlap (round 1)'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', choices=['b200', 'reference'], default='b200')
    ap.add_argument('--workload', choices=list(WORKLOADS), default='c2')
    ap.add_argument('--basins', type=int, default=None, help='override basins per GPU')
    ap.add_argument('--ckpt', type=int, default=0, choices=[0, 1, 2, 4, 8, 16, 32],
                    help='checkpoint interval of the adjoint (0 = library default: 1 for small problems, else 16)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-at-scale', action='store_true')
    ap.add_argument('--no-configs', action='store_true', help='skip BASELINE configs 4 and 5 in at_scale')
    ap.add_argument('--no-cpu-slices', action='store_true', help='skip the CPU slices of configs 3-5 in cpu_baseline')
    ap.add_argument('--no-graph', dest='graph', action='store_false',
                    help='time the eager step instead of a CUDA-graph replay of it (single GPU: the step '
                         'is ~0.55 ms of kernels, about what one eager Python step costs the host, so the '
                         'eager number depends on the host CPU; with several GPUs the all-reduce runs '
                         'eagerly after each replay)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one returned (every output series, the loss, '
                         'the parameter gradient; rank 0) as DIR/<name>.npy in float32, at most 64 MB in all: '
                         'beyond that a fixed, seeded subset of basins')
    ap.set_defaults(graph=True)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(3, args.warmup)
    # stdout carries exactly one JSON line: while the run is in progress file descriptor 1 points at
    # stderr (library banners written by native code land there), the line goes to the real stdout
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)
    if args.impl == 'reference':
        return run_reference(args)
    return run_b200(args)


_REAL_STDOUT = None


def emit(line: dict) -> None:
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + '\n')
    out.flush()


if __name__ == '__main__':
    sys.exit(main())
