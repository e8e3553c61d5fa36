"""F-estimation distances, GPU (jb_dist_*, csrc/distances.cuh) against the host path (sklearn / scipy), at single-cell sizes.

    python tools/dist_bench.py [--out DIR] [--host-max 2e11] [--only NAME ...]

For every workload (fixed seeds): GPU wall time per phase, each ending in a device synchronise -- accumulate (host slab
preparation, host-to-device copies and the accumulation kernels, overlapped, plus the finishing transform), kNN selection,
all-pairs shortest paths (graph build + blocked Floyd-Warshall + unreachable rule) and copy-out of the n x n float64
matrix -- the host path's time (skipped when n^2 d exceeds --host-max, and said so), the agreement of the two outputs, and
rates against the data-sheet fp64 figure. One workload is then re-run under torch.profiler for the kernel-only times.
Writes DIR/dist_bench.json and prints a markdown table.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from jamie_b200 import correspondence as CR  # noqa: E402

# HGX B200 data sheet: 37 TFLOP/s fp64 per GPU (296 for eight) at up to 1000 W = 18.5e12 fma/s. A pair-column update of
# the accumulation is one fma (plus a subtraction for the difference forms); a Floyd-Warshall relaxation is one add and
# one min, so its bound is taken as 18.5e12 relaxations/s too.
FP64_FMA_PEAK = 18.5e12


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else 'unknown'
    except Exception as e:   # noqa: BLE001
        return f'unknown ({e})'


def make(kind, n, d, seed):
    rng = np.random.default_rng(seed)
    if kind == 'clusters':     # six well separated clusters: the kNN graph never connects, k climbs to its cap
        centres = rng.standard_normal((6, d)) * 20
        X = centres[np.arange(n) % 6] + rng.standard_normal((n, d), dtype=np.float32)
        return X.astype(np.float32)
    if kind == 'manifold':     # one noisy curve: connected at a small k
        t = np.sort(rng.random(n)) * 10
        lat = np.stack([np.cos(t) * t, np.sin(t) * t, t, np.cos(2 * t)], 1)
        X = lat @ rng.standard_normal((4, d)) + 0.05 * rng.standard_normal((n, d), dtype=np.float32)
        return X.astype(np.float32)
    if kind == 'counts':       # non-negative, offset like log counts
        return (rng.standard_normal((n, d), dtype=np.float32) + 3.0).clip(0)
    if kind == 'sparse':
        import scipy.sparse as sp
        nnz = int(0.02 * n * d)
        rows, cols = np.repeat(np.arange(n), nnz // n), rng.integers(0, d, n * (nnz // n))
        vals = rng.random(len(rows), dtype=np.float32) * 4
        return sp.csr_matrix((vals, (rows, cols)), shape=(n, d))
    raise ValueError(kind)


WORKLOADS = [
    # name, mode, data kind, n, d
    ('geo_clusters_9000x2000', 'geodesic', 'clusters', 9000, 2000),
    ('geo_manifold_9000x2000', 'geodesic', 'manifold', 9000, 2000),
    ('geo_manifold_20000x2000', 'geodesic', 'manifold', 20000, 2000),
    ('geo_counts_9190x28930', 'geodesic', 'counts', 9190, 28930),
    ('euclidean_20000x28930', 'euclidean', 'counts', 20000, 28930),
    ('pearson_20000x28930', 'pearson', 'counts', 20000, 28930),
    ('geo_sparse_9190x241757_2pct', 'geodesic', 'sparse', 9190, 241757),
]


def run_gpu(X, mode, kmax=40):
    """gpu_distance_function's steps with a synchronised clock around each phase"""
    n, d = X.shape
    kind, prep, transform = CR.GPU_DISTANCE_MODES[mode]
    t = {}
    m = CR.DeviceDistances(n, 0)
    try:
        t0 = time.perf_counter()
        for slab in CR.prepared_slabs(X, prep, max(1, min(d, CR.SLAB_BYTES // (8 * n)))):
            m.accumulate(kind, slab)
        m.finish(transform, copy=False)
        t['accumulate'] = time.perf_counter() - t0
        k = None
        if mode == 'geodesic':
            t0 = time.perf_counter()
            idx, _ = m.knn(CR.knn_list_width(n, kmax))
            t['select'] = time.perf_counter() - t0
            t0 = time.perf_counter()
            k = min(CR.connectivity_k(idx, kmax), n)
            t['connectivity_loop_host'] = time.perf_counter() - t0
            t0 = time.perf_counter()
            m.geodesic(k, copy=False)
            t['apsp'] = time.perf_counter() - t0
        t0 = time.perf_counter()
        out = m.finish(0)      # transform 0: no kernel, the copy-out alone
        t['copy_out'] = time.perf_counter() - t0
    finally:
        m.close()
    return out, t, k


def kernel_profile(X, mode):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_gpu(X, mode)
        torch.cuda.synchronize()
    agg = {}
    for ev in prof.key_averages():
        if ev.device_type is not None and 'CUDA' in str(ev.device_type) and ev.self_device_time_total > 0:
            agg[ev.key] = (agg.get(ev.key, (0, 0))[0] + ev.self_device_time_total / 1e6, ev.count)
    return {k: {'seconds': round(v[0], 4), 'launches': v[1]} for k, v in sorted(agg.items(), key=lambda kv: -kv[1][0])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='.', help='directory of dist_bench.json')
    ap.add_argument('--host-max', type=float, default=2e11, help='skip the host path above this n^2 d')
    ap.add_argument('--only', nargs='*')
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), 'dist_bench measures the GPU path: it needs a CUDA device'
    info = {'gpu': gpu_info(), 'torch_device': torch.cuda.get_device_name(0), 'host_cpus': os.cpu_count(), 'workloads': []}
    print('GPU (name, power limit, max SM clock):', info['gpu'], '| host CPUs:', info['host_cpus'], flush=True)
    for name, mode, kind, n, d in WORKLOADS:
        if args.only and name not in args.only:
            continue
        t0 = time.perf_counter()
        X = make(kind, n, d, seed=len(name))
        gen = time.perf_counter() - t0
        out, t, k = run_gpu(X, mode)
        rec = {'name': name, 'mode': mode, 'n': n, 'd': d, 'data_seconds': round(gen, 2), 'k': k,
               'gpu_seconds': {p: round(v, 4) for p, v in t.items()}, 'gpu_total': round(sum(t.values()), 3)}
        rec['accumulate_fma_per_s'] = n * n * d / 2 / t['accumulate']
        rec['accumulate_share_of_fp64_peak'] = rec['accumulate_fma_per_s'] / FP64_FMA_PEAK
        if 'apsp' in t:
            rec['apsp_relax_per_s'] = float(n) ** 3 / t['apsp']
            rec['apsp_share_of_fp64_peak'] = rec['apsp_relax_per_s'] / FP64_FMA_PEAK
        if float(n) * n * d <= args.host_max:
            dense = X.toarray() if hasattr(X, 'toarray') else X
            t0 = time.perf_counter()
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                host = CR.distance_function(mode, 40)(dense)
            rec['host_seconds'] = round(time.perf_counter() - t0, 2)
            diff = np.abs(out.astype(np.float64) - host)
            rec['max_abs_diff_over_scale'] = float(np.nanmax(diff) / np.nanmax(np.abs(host)))
            rec['max_rel_diff'] = float(np.nanmax(diff / np.maximum(np.abs(host), 1e-300)))
            rec['speedup'] = round(rec['host_seconds'] / rec['gpu_total'], 1)
        else:
            rec['host_seconds'] = f'skipped (n^2 d = {float(n) * n * d:.2e} > {args.host_max:.0e})'
        print(json.dumps(rec), flush=True)
        info['workloads'].append(rec)
        del out, X
    if not args.only or WORKLOADS[0][0] in args.only:
        name, mode, kind, n, d = WORKLOADS[0]
        info['kernel_profile'] = {'workload': name, 'kernels': kernel_profile(make(kind, n, d, seed=len(name)), mode)}
        print(json.dumps(info['kernel_profile']), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, 'dist_bench.json'), 'w') as f:
        json.dump(info, f, indent=1)
    print('\n| workload | k | accumulate s | select s | APSP s | copy-out s | GPU total s | host s | agreement (max |diff| / scale) |')
    print('|---|---|---|---|---|---|---|---|---|')
    for r in info['workloads']:
        g = r['gpu_seconds']
        print(f"| {r['name']} | {r['k']} | {g['accumulate']:.3f} | {g.get('select', '-')} | {g.get('apsp', '-')} | {g['copy_out']:.3f} | "
              f"{r['gpu_total']:.3f} | {r['host_seconds']} | {r.get('max_abs_diff_over_scale', '-')} |")


if __name__ == '__main__':
    main()
