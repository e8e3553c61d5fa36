"""The benchmark's JSON contract on a real GPU (short run): one line on stdout, the keys the driver reads, sane values."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_line_contract(tmp_path):
    dump = tmp_path / 'outputs'
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '60', '--warmup', '5', '--no-cpu-baseline', '--no-fit',
                          '--dump-outputs', str(dump)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d['metric'].startswith('train cells/sec') and d['unit'] == 'cells/s' and d['n_gpus'] == 1
    assert d['steps'] == 60 and d['warmup'] == 5 and d['higher_is_better'] is True and d['scaling'] == 'weak'
    assert d['value'] > 1e5 and abs(d['value'] - 512 / (d['ms_per_step'] * 1e-3)) < 1e-6 * d['value']
    assert d['vs_baseline'] is None and d['data'] == 'synthetic' and 'workload' in d['config']
    e = d['e2e']
    assert 0 < e['value'] <= 1.05 * d['value'] and e['h2d_bytes_per_step'] > 2 * 512 * 512 * 4 and e['d2h_bytes_per_step'] == 32
    # the 60 timed steps are ONE launch of the persistent step kernel (+ the barrier-counter reset node is a memset, and the
    # one-thread control-block update kernel): 2 kernel launches
    assert d['gpu_launches'] >= 1 and abs(d['gpu_launches'] - d['launches_per_step'] * 60) < 1e-6
    r = d['roofline']
    assert r['bound'] == 'hbm' and 0 < r['frac'] < 1 and abs(r['frac'] - r['achieved'] / r['peak']) < 1e-9
    assert r['traffic'] is None or r['traffic'] > 0
    g = d['gemm_roofline']
    assert g['bound'] == 'tensor' and 0 < g['frac'] < 1
    names = [nm for nm, _ in d['step_profile']['phases']]
    assert 'adam' in names and 'wgrad x12' in names and abs(d['step_profile']['sum_us'] - d['ms_per_step'] * 1e3) < 0.25 * d['ms_per_step'] * 1e3
    assert set(d['clocks']) >= {'sm_mhz', 'sm_max_mhz', 'reasons'}
    p = d['modal_predict']
    assert p['value'] > 1e6 and p['e2e']['value'] > 1e5 and 0 < p['roofline']['frac'] < 1
    assert all(k in d['final_losses'] for k in ('KL', 'Rec', 'CosSim', 'F', 'total', 'grad_norm'))
    # --dump-outputs: the last timed step's results, float32, the reference's packed orders
    from jamie_b200.layout import bn_spec, param_spec
    files = {f.stem: np.load(f) for f in dump.glob('*.npy')}
    n_params = sum(int(np.prod(s)) for _, s in param_spec([512, 512], 32))
    shapes = {'losses': (6,), 'grads': (n_params,), 'params': (n_params,), 'bn_stats': (2 * sum(w for _, w in bn_spec([512, 512])),)}
    assert {k: a.shape for k, a in files.items()} == shapes
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in files.values())
    assert sum(f.stat().st_size for f in dump.iterdir()) <= 64 << 20
    assert files['losses'].tolist() == [d['final_losses'][k] for k in ('KL', 'Rec', 'CosSim', 'F', 'total', 'grad_norm')]


def test_bench_dump_is_the_last_timed_step_and_reproducible(tmp_path):
    """Two runs with the same arguments dump bit-identical outputs; the dump is the trained state after the timed steps
    (not the initial weights / BatchNorm statistics) and its gradients are those whose norm the last timed step reported."""
    from bench import init_params
    dumps = []
    for run in ('a', 'b'):
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '8', '--warmup', '3', '--no-cpu-baseline',
                              '--no-fit', '--no-predict', '--dump-outputs', str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-3000:]
        dumps.append({f.stem: np.load(f) for f in (tmp_path / run).glob('*.npy')})
    a, b = dumps
    assert sorted(a) == sorted(b) == ['bn_stats', 'grads', 'losses', 'params']
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    params, bufs = init_params()
    init = np.concatenate([p.ravel() for p in params])
    assert np.mean(a['params'] != init) > 0.5
    bn_init = np.concatenate([v for k, v in bufs.items() if not k.endswith('.num_batches_tracked')])
    assert np.mean(a['bn_stats'] != bn_init) > 0.5
    assert abs(np.linalg.norm(a['grads'].astype(np.float64)) - a['losses'][5]) < 1e-4 * a['losses'][5]
