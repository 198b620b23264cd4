"""bench.py contract checks: the reference arm prints exactly one JSON line with the keys a reader
of the bench line relies on, the B200 arm refuses to run without a CUDA device (no CPU path), and
--dump-outputs writes the last timed step's results (the B200 arm's on the GPU)."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import RTOL_GRAD, assert_close, assert_grad_close, flux_rtol

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1',
                        '--warmup', '3', '--basins', '4'], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'basin-timesteps/s' and d['higher_is_better'] is True
    assert d['metric'].startswith('basin-timesteps/sec') and d['dtype'] == 'f32' and d['vs_baseline'] is None
    # the same `config` as the B200 arm prints (same workload, full size, every step); what ran on
    # the CPU — the unmodified reference from baseline/_ref, else the oracle port — is in cpu_baseline
    assert 'workload' in d['config'] and d['config']['basins_per_gpu'] == 4 and 'sample' in d['cpu_baseline']
    have_ref = os.path.isdir(os.path.join(ROOT, 'baseline', '_ref', 'hydrodl2'))
    assert d['cpu_baseline']['kind'] == ('reference' if have_ref else 'port') and d['cpu_baseline']['cores'] >= 1
    assert d['cpu_baseline']['value'] == d['value'] == d['e2e']['value'] > 0
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0


def test_b200_arm_needs_cuda():
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '1'],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and r.stdout.strip() == ''
    assert 'no CPU fallback' in r.stderr


def _oracle_step(basins):
    """One training step of the bench workload on the CPU oracle, on bench.py's own inputs."""
    import bench
    from oracle import hbv_oracle as O
    wl = bench.WORKLOADS['c2']
    x, p = bench.make_inputs(wl, basins, bench.SEED)
    pc = p.clone().requires_grad_(True)
    out, _ = O.forward_packed(wl['model'], x, pc, nmul=bench.NMUL, warm_up=wl['warm_up'], dynamic_params=wl['dyn'])
    out['streamflow'].sum().backward()
    return out, pc.grad


def _load_dump(d):
    arrays = {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}
    for k, a in arrays.items():
        assert a.dtype == np.float32, k
    return {k: torch.from_numpy(a) for k, a in arrays.items()}


def _bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), *args], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert len([ln for ln in r.stdout.splitlines() if ln.strip()]) == 1, r.stdout
    return json.loads(r.stdout)


def test_reference_arm_dumps_the_last_step(tmp_path):
    """Plumbing of --dump-outputs: the dump holds every output, the loss and the gradient of the
    last timed step on bench.py's inputs.  Without baseline/_ref the arm runs the oracle port, so
    this compares the oracle with itself and checks no numerics; the B200 arm's test below does."""
    d = str(tmp_path / 'out')
    _bench('--impl', 'reference', '--steps', '1', '--warmup', '3', '--basins', '3', '--dump-outputs', d)
    got = _load_dump(d)
    out, grad = _oracle_step(3)
    assert set(got) == set(out) | {'loss', 'grad_parameters'}
    for k, v in out.items():
        assert_close(got[k], v, 1e-6, f'dumped {k}')
    assert_close(got['grad_parameters'], grad, 1e-6, 'dumped grad_parameters')
    assert_close(got['loss'], out['streamflow'].sum(), 1e-6, 'dumped loss')


def test_dump_outputs_samples_basins_within_the_limit(tmp_path):
    """An output set larger than the limit keeps the same seeded basins in every per-basin array
    (each entry here holds its basin's index), every time."""
    import bench
    T, B, ncol = 1095, 600, 210
    basin = torch.arange(B, dtype=torch.float32)
    out = {'streamflow': basin.view(1, B, 1).expand(T, B, 1), 'BFI': basin}
    grad = basin.view(1, B, 1).expand(T, B, ncol)      # 550 MB if materialised
    kept = []
    for run in ('a', 'b'):
        d = str(tmp_path / run)
        bench.dump_outputs(d, out, torch.tensor(1.5), grad, torch.ones(ncol))
        assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= bench.DUMP_LIMIT
        got = _load_dump(d)
        assert set(got) == {'streamflow', 'BFI', 'loss', 'grad_parameters', 'grad_shared'}
        idx = got['BFI']
        assert 0 < len(idx) < B and bool((idx[1:] > idx[:-1]).all())
        assert torch.equal(got['streamflow'], idx.view(1, -1, 1).expand(T, -1, 1))
        assert torch.equal(got['grad_parameters'], idx.view(1, -1, 1).expand(T, -1, ncol))
        assert got['loss'].item() == 1.5 and torch.equal(got['grad_shared'], torch.ones(ncol))
        kept.append(idx)
    assert torch.equal(kept[0], kept[1])


@pytest.mark.gpu
def test_b200_arm_dumps_the_last_step(tmp_path):
    """The B200 arm's dump is the bench step's result: it matches the CPU oracle on the same inputs."""
    d = str(tmp_path / 'out')
    line = _bench('--steps', '2', '--warmup', '3', '--basins', '8', '--no-cpu-baseline', '--dump-outputs', d)
    assert line['steps'] == 2
    got = _load_dump(d)
    out, grad = _oracle_step(8)
    assert set(got) == set(out) | {'loss', 'grad_parameters', 'grad_shared'}
    for k, v in out.items():
        assert_close(got[k], v, flux_rtol(k), f'dumped {k}')
    assert_grad_close(got['grad_parameters'], grad, 'dumped grad_parameters', 16)
    assert_close(got['loss'], out['streamflow'].sum(), flux_rtol('streamflow'), 'dumped loss')
    assert_close(got['grad_shared'], got['grad_parameters'][-1].sum(0), RTOL_GRAD, 'dumped grad_shared')
