"""Silhouette coefficients (evaluation.silhouette_samples: jb_silhouette) against FOSCTTM's tile work at the same size and
against sklearn's silhouette_samples on the host.

  python tools/silhouette_bench.py [--quick] [--sizes N,N,...] [--host-sizes N,N,...] [--out FILE.md] [--trace-dir DIR]

Cases: L = 32 standard normal rows, n = 10^5 and 10^6, C = 2, 20 and 1 000 labels of random sizes (each row's label
drawn uniformly).
  device : the whole silhouette_samples call (label encoding and sort on the host, the jb_silhouette call: row upload,
           k_sil_partial, k_sil_finish, sums back, sklearn's finish) and jb_metric_foscttm on two [n, 32] embeddings:
           the same n^2 float64 tile arithmetic with a counting consumer, so the ratio of the two is the cost of the
           per-pair sqrt and the label-segment sums.
  host   : sklearn.metrics.silhouette_samples at --host-sizes (float64 rows); the time per pair there extrapolates to
           the device sizes, marked as such.
Times are medians of 3 calls after one warm-up (one call, no warm-up beyond a small one, for n = 10^6), each ending in
a synchronise; device phases come from a separate torch.profiler run of one call at n <= 10^5.
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

L = 32


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def median_time(fn, reps=3):
    if reps > 1:
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
        prof.export_chrome_trace(os.path.join(trace_dir, f'silhouette_{tag}.json'))
    out = {}
    for ev in prof.key_averages():
        us = getattr(ev, 'device_time_total', None)
        us = ev.cuda_time_total if us is None else us
        for key, ph in (('k_sil_partial', 'partial'), ('k_sil_finish', 'finish'), ('k_foscttm', 'foscttm'),
                        ('HtoD', 'copy H2D'), ('DtoH', 'copy D2H')):
            if key in ev.key:
                out[ph] = out.get(ph, 0.0) + us / 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--quick', action='store_true')
    ap.add_argument('--sizes', default=None)
    ap.add_argument('--host-sizes', default=None)
    ap.add_argument('--out', default=None)
    ap.add_argument('--trace-dir', default=None)
    a = ap.parse_args()
    sizes = [int(s) for s in a.sizes.split(',')] if a.sizes else ([20000] if a.quick else [100000, 1000000])
    host_sizes = [int(s) for s in a.host_sizes.split(',')] if a.host_sizes else ([2000] if a.quick else [10000, 30000])
    import torch
    from jamie_b200 import _lib
    from jamie_b200.evaluation import silhouette_samples
    from sklearn.metrics import silhouette_samples as sk_samples
    lib = _lib.load()
    if a.trace_dir:
        os.makedirs(a.trace_dir, exist_ok=True)
    gpu = card()
    print(gpu, flush=True)
    p = lambda x: x.ctypes.data_as(C.c_void_p)   # noqa: E731

    host_lines = ['', '## Host: sklearn.metrics.silhouette_samples (L = 32, 20 labels, float64 rows)', '',
                  '| n | sklearn s | ns per pair | device silhouette_samples s | max abs difference |', '|---|---|---|---|---|']
    ns_pair = None
    for n in host_sizes:
        rng = np.random.default_rng(n)
        X = rng.standard_normal((n, L)).astype(np.float32).astype(np.float64)
        labels = rng.integers(0, 20, n)
        silhouette_samples(X[:1000], labels[:1000])
        t0 = time.perf_counter()
        want = sk_samples(X, labels)
        t_host = time.perf_counter() - t0
        t0 = time.perf_counter()
        got = silhouette_samples(X, labels)
        t_dev = time.perf_counter() - t0
        ns_pair = t_host / n ** 2 * 1e9
        host_lines.append(f'| {n} | {t_host:.2f} | {ns_pair:.2f} | {t_dev:.3f} | {np.abs(got - want).max():.1e} |')
        print(host_lines[-1], flush=True)

    lines = [f'# Silhouette coefficients on {gpu}', '',
             'Card name and power limit from nvidia-smi in the same command as the measurements. Times in seconds '
             '(median of the calls; one call at n = 10^6), device phases in ms from one profiled call (n <= 10^5).', '',
             '## Device (L = 32)', '',
             '| n | labels | silhouette_samples s | k_sil_partial ms | k_sil_finish ms | H2D ms | D2H ms | FOSCTTM call s | '
             'FOSCTTM kernel ms | silhouette / FOSCTTM call | sklearn s (extrapolated, not run) |',
             '|---|---|---|---|---|---|---|---|---|---|---|']
    for n in sizes:
        rng = np.random.default_rng(n)
        X = rng.standard_normal((n, L), dtype=np.float32)
        Y = rng.standard_normal((n, L), dtype=np.float32)
        reps = 1 if n >= 1000000 else 3
        prof = n <= 100000
        cnt = C.c_ulonglong(0)

        def fos(rows=n):
            _lib.check(lib.jb_metric_foscttm(p(X), p(Y), rows, L, 0, C.byref(cnt)))
        if reps == 1:
            fos(5000)   # module load and first-launch costs outside the single timed call
        t_fos = median_time(fos, reps)
        ph_fos = phases(fos, a.trace_dir, f'foscttm_{n}') if prof else {}
        for n_labels in (2, 20, 1000):
            labels = rng.integers(0, n_labels, n)
            if reps == 1:
                silhouette_samples(X[:5000], labels[:5000])
            t_s = median_time(lambda: silhouette_samples(X, labels), reps)
            ph = phases(lambda: silhouette_samples(X, labels), a.trace_dir, f'{n}_{n_labels}') if prof else {}
            ext = 'not measured' if ns_pair is None else f'{ns_pair * n ** 2 / 1e9:.0f}'
            g = lambda d, k: f'{d[k]:.1f}' if k in d else 'not measured'   # noqa: E731
            lines.append(f'| {n} | {n_labels} | {t_s:.3f} | {g(ph, "partial")} | {g(ph, "finish")} | {g(ph, "copy H2D")} | '
                         f'{g(ph, "copy D2H")} | {t_fos:.3f} | {g(ph_fos, "foscttm")} | {t_s / t_fos:.2f} | {ext} |')
            print(lines[-1], flush=True)
        torch.cuda.synchronize()
    text = '\n'.join(lines + host_lines) + '\n'
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(text)


if __name__ == '__main__':
    main()
