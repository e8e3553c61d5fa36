"""Exact kNN search and kNN imputation (evaluation.kneighbors / knn_impute: jb_knn, jb_knn_average) against FOSCTTM's
tile work at the same size and against sklearn's brute-force estimators on the host.

  python tools/knn_bench.py [--quick] [--sizes N,N,...] [--host-max N] [--out FILE.md] [--trace-dir DIR]

Cases: L = 32 embeddings, nq = nr = n for n = 10^4, 10^5, 10^6, k = 5 and 50.
  search : the jb_knn call (reference and query upload, k_knn_search, k_knn_merge, lists back), and
           jb_metric_foscttm on two [n, 32] embeddings: the same n^2 float64 tile arithmetic with a counting consumer,
           so the ratio of the two is the cost of the selection.
  average: jb_knn_average on dense float64 values [n, 2 000], and the whole knn_impute with a scipy.sparse CSR [n, 34 861]
           at 5 % density (host CSC conversion and per-slab densification included).
  host   : sklearn NearestNeighbors(algorithm='brute').kneighbors and KNeighborsRegressor(algorithm='brute') on the dense
           values, for n <= --host-max; larger sizes are "not measured".
Times are medians of 3 calls after one warm-up (one call for n = 10^6; the sparse knn_impute: one call after a profiled
one), each ending in a synchronise; device phases come from a separate torch.profiler run of one call. The host
regressor and the sparse case run at k = 50 only for n = 10^4, to keep the run within minutes. Embeddings are standard
normal; the values' contents do not change the timing.
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

D_DENSE, D_SPARSE, DENSITY, L = 2000, 34861, 0.05, 32


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def median_time(fn, reps=3):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def phases(fn, trace_dir, tag):
    """Device time per phase (ms) of one profiled call, by kernel / copy name."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    if trace_dir:
        prof.export_chrome_trace(os.path.join(trace_dir, f'knn_{tag}.json'))
    out = {}
    for ev in prof.key_averages():
        us = getattr(ev, 'device_time_total', None)
        us = ev.cuda_time_total if us is None else us
        name = ev.key
        for key, ph in (('k_knn_search', 'search'), ('k_knn_merge', 'merge'), ('k_knn_average', 'average'),
                        ('k_foscttm', 'foscttm'), ('HtoD', 'copy H2D'), ('DtoH', 'copy D2H')):
            if key in name:
                out[ph] = out.get(ph, 0.0) + us / 1e3
    return out


def sparse_values(n, rng):
    per = int(D_SPARSE * DENSITY)
    indptr = np.arange(n + 1, dtype=np.int64) * per
    indices = np.sort(rng.integers(0, D_SPARSE, (n, per), dtype=np.int32), axis=1).ravel()
    import scipy.sparse as sp
    return sp.csr_matrix((np.ones(n * per), indices, indptr), shape=(n, D_SPARSE))


def fmt(t):
    return 'not measured' if t is None else f'{t:.3f}'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--quick', action='store_true')
    ap.add_argument('--sizes', default=None)
    ap.add_argument('--host-max', type=int, default=100000)
    ap.add_argument('--out', default=None)
    ap.add_argument('--trace-dir', default=None)
    a = ap.parse_args()
    sizes = [int(s) for s in a.sizes.split(',')] if a.sizes else ([2000, 20000] if a.quick else [10000, 100000, 1000000])
    import torch
    from jamie_b200 import _lib, evaluation
    from jamie_b200.evaluation import DeviceKnn
    lib = _lib.load()
    if a.trace_dir:
        os.makedirs(a.trace_dir, exist_ok=True)
    gpu = card()
    lines = [f'# kNN search and kNN imputation on {gpu}', '',
             'Card name and power limit from nvidia-smi in the same command as the measurements. Times in seconds '
             '(median of the calls), device phases in ms from one profiled call.', '',
             '## Search (L = 32, nq = nr = n)', '',
             '| n | k | jb_knn call s | search ms | merge ms | H2D ms | D2H ms | FOSCTTM call s | FOSCTTM kernel ms | search / FOSCTTM call | sklearn kneighbors s |',
             '|---|---|---|---|---|---|---|---|---|---|---|']
    avg_lines = ['', '## Average (k = 5 and 50 neighbour lists from the search above)', '',
                 '| n | k | values | call s | average ms | H2D ms | D2H ms | sklearn KNeighborsRegressor s |',
                 '|---|---|---|---|---|---|---|---|']
    print(gpu, flush=True)
    for n in sizes:
        rng = np.random.default_rng(n)
        q = rng.standard_normal((n, L), dtype=np.float32)
        r = rng.standard_normal((n, L), dtype=np.float32)
        reps = 1 if n >= 1000000 else 3
        cnt = C.c_ulonglong(0)
        p = lambda x: x.ctypes.data_as(C.c_void_p)   # noqa: E731

        def fos():
            _lib.check(lib.jb_metric_foscttm(p(q), p(r), n, L, 0, C.byref(cnt)))
        t_fos = median_time(fos, reps)
        ph_fos = phases(fos, a.trace_dir, f'foscttm_{n}')
        Vd = np.ones((n, D_DENSE)) if n >= 1000000 else rng.random((n, D_DENSE))
        Vs = sparse_values(n, rng) if n <= 100000 else None
        for k in (5, 50):
            res = {}

            def search():
                res['lists'] = DeviceKnn.search(q, r, k, evaluation.KNN_BATCH_BYTES, None)
            t_s = median_time(search, reps)
            ph = phases(search, a.trace_dir, f'search_{n}_{k}')
            t_host = None
            if n <= a.host_max:
                from sklearn.neighbors import NearestNeighbors
                nn = NearestNeighbors(n_neighbors=k, algorithm='brute').fit(r)
                t0 = time.perf_counter()
                _, si = nn.kneighbors(q)
                t_host = time.perf_counter() - t0
                print(f'  n={n} k={k}: sklearn index agreement {np.mean(si == res["lists"][1]):.6f}', flush=True)
            ratio = t_s / t_fos
            lines.append(f'| {n} | {k} | {t_s:.3f} | {ph.get("search", 0):.1f} | {ph.get("merge", 0):.2f} | '
                         f'{ph.get("copy H2D", 0):.1f} | {ph.get("copy D2H", 0):.1f} | {t_fos:.3f} | '
                         f'{ph_fos.get("foscttm", 0):.1f} | {ratio:.2f} | {fmt(t_host)} |')
            print(lines[-1], flush=True)
            _, idx = res['lists']

            def avg():
                DeviceKnn.average(idx, None, Vd, evaluation.KNN_BATCH_BYTES, None)
            t_a = median_time(avg, reps)
            pa = phases(avg, a.trace_dir, f'average_{n}_{k}')
            t_hr = None
            if n <= a.host_max and (k == 5 or n <= 10000):
                from sklearn.neighbors import KNeighborsRegressor
                reg = KNeighborsRegressor(n_neighbors=k, algorithm='brute').fit(r, Vd)
                t0 = time.perf_counter()
                reg.predict(q)
                t_hr = time.perf_counter() - t0
            avg_lines.append(f'| {n} | {k} | dense [n, {D_DENSE}] | {t_a:.3f} | {pa.get("average", 0):.1f} | '
                             f'{pa.get("copy H2D", 0):.1f} | {pa.get("copy D2H", 0):.1f} | {fmt(t_hr)} |')
            print(avg_lines[-1], flush=True)
            if Vs is not None and (k == 5 or n <= 10000):
                pi = phases(lambda: evaluation.knn_impute(q, r, Vs, k=k), a.trace_dir, f'impute_sparse_{n}_{k}')
                t0 = time.perf_counter()
                evaluation.knn_impute(q, r, Vs, k=k)
                t_i = time.perf_counter() - t0
                avg_lines.append(f'| {n} | {k} | knn_impute, CSR [n, {D_SPARSE}] 5 % | {t_i:.3f} | '
                                 f'{pi.get("average", 0):.1f} | {pi.get("copy H2D", 0):.1f} | {pi.get("copy D2H", 0):.1f} | '
                                 'not measured |')
            else:
                avg_lines.append(f'| {n} | {k} | knn_impute, CSR [n, {D_SPARSE}] 5 % | not measured | not measured | '
                                 'not measured | not measured | not measured |')
            print(avg_lines[-1], flush=True)
        del Vd, Vs
        torch.cuda.synchronize()
    text = '\n'.join(lines + avg_lines) + '\n'
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(text)


if __name__ == '__main__':
    main()
