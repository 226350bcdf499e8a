"""bench.py contract checks that need no GPU: the reference arm (the reference graph over the oracle port on the host CPU) prints one
JSON line with the agreed keys; ranks other than 0 print nothing and exit 0; our arm refuses to run without a CUDA device."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + args, capture_output=True, text=True, timeout=timeout,
                          env=dict(os.environ, **(env or {})))


def test_reference_arm_prints_one_json_line():
    r = _run(['--impl', 'reference', '--cpu-batch', '1', '--steps', '1', '--warmup', '1'])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'train_meshes_per_sec' and d['unit'] == 'meshes/s' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': 'meshes/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'workload' in d['config'] and d['vs_baseline'] is None


def test_reference_arm_uses_all_cores_and_never_maps_the_product_library():
    """Under torchrun OMP_NUM_THREADS=1 is exported: the arm must still use every host core.  It runs oracle/ only, so neither the
    product package nor libgeniconet_b200.so may appear in the process."""
    code = ("import os, sys, json; sys.path.insert(0, %r); import bench; "
            "t, threads = bench.cpu_reference_step_time('ico2ico', 5, 1, 1, 0); "
            "maps = open('/proc/self/maps').read(); "
            "print(json.dumps({'threads': threads, 'so': 'libgeniconet' in maps, "
            "'mods': [m for m in sys.modules if m.startswith('geniconet_b200')]}))" % ROOT)
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=600, env=dict(os.environ, OMP_NUM_THREADS='1'))
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d['threads'] == (os.cpu_count() or 1) and not d['so'] and not d['mods'], d


def test_reference_arm_other_ranks_exit_quietly():
    r = _run(['--impl', 'reference', '--gpus', '2'], env={'RANK': '1', 'WORLD_SIZE': '2', 'LOCAL_RANK': '1'})
    assert r.returncode == 0 and r.stdout.strip() == ''


def test_our_arm_has_no_cpu_path():
    import torch
    if torch.cuda.is_available():
        pytest.skip('a CUDA device is present')
    r = _run(['--steps', '1', '--warmup', '1', '--no-cpu-baseline'])
    assert r.returncode != 0 and 'no CUDA device' in (r.stderr + r.stdout)


def test_steps_must_be_positive():
    r = _run(['--steps', '0', '--no-cpu-baseline'])
    assert r.returncode != 0 and '--steps must be at least 1' in r.stderr
    r = _run(['--impl', 'reference', '--dump-outputs', 'unused'])
    assert r.returncode != 0 and '--dump-outputs' in r.stderr


def test_reference_arm_times_the_requested_steps():
    r = _run(['--impl', 'reference', '--cpu-batch', '1', '--level', '3', '--steps', '6', '--warmup', '2'])
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d['steps'] == 6 and d['warmup'] == 2


def _dump(tmp_path, tag, *extra):
    import numpy as np
    out = tmp_path / tag
    r = _run(['--steps', '3', '--warmup', '1', '--no-cpu-baseline', '--no-kernel-table', '--dump-outputs', str(out)] + list(extra))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])['steps'] == 3
    assert sum(f.stat().st_size for f in out.iterdir()) <= (64 << 20) + 256 * len(list(out.iterdir()))     # + .npy headers
    return {f.name[:-4]: np.load(f) for f in out.iterdir()}


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_step(tmp_path):
    """--dump-outputs: inputs, loss, output, parameters and gradients of the last timed step as float32 .npy files; two runs with
    the same arguments dump the same inputs and (up to reordered float sums) the same results."""
    import numpy as np
    from geniconet_b200 import models as gm
    a, b = _dump(tmp_path, 'a'), _dump(tmp_path, 'b')
    assert sorted(a) == sorted(b) and all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    names = [n for n, _ in gm.ico2ico(gm.default_params('ico2ico')).named_parameters()]
    assert sorted(k for k in a if k.startswith('param.')) == sorted('param.' + n for n in names)
    assert sorted(k for k in a if k.startswith('grad.')) == sorted('grad.' + n for n in names)
    assert a['loss'].shape == (1,) and a['output'].shape == (36, 3, 160, 64) and a['input.x'].shape == (36, 3, 160, 64)
    assert np.abs(a['grad.encoder.0.weight']).max() > 0
    for k in ('input.x', 'input.target'):
        assert np.array_equal(a[k], b[k]), k
    for k in a:
        assert np.allclose(a[k], b[k], rtol=1e-4, atol=1e-6 * max(1.0, float(np.abs(a[k]).max()))), k


@pytest.mark.gpu
def test_dump_outputs_samples_large_arrays(tmp_path):
    """ico2ico_vae at batch 72: the arrays exceed the 64 MB budget, so the reconstruction and the input are stored as seeded samples."""
    v = _dump(tmp_path, 'vae', '--model', 'ico2ico_vae', '--batch', '72')
    assert {'loss', 'output', 'mu', 'logvar', 'input.x', 'input.target'} <= set(v)
    # the reconstruction (72 x 3 x 160 x 64) is above every cap the budget allows: it is sampled down to the cap, and no array is
    # larger than that cap; the input has the same size, so it is sampled to the same number of elements
    cap = v['output'].size
    assert v['output'].ndim == 1 and cap < 72 * 3 * 160 * 64
    assert v['input.x'].ndim == 1 and v['input.x'].size == cap
    assert all(a.size <= cap for a in v.values()) and v['mu'].size == v['logvar'].size
