"""Per-feature AUROC (evaluation.imputation_auroc, jb_metric_feature_auroc) against the roc_auc_score loop it replaces.

  python tools/auroc_bench.py [--quick] [--out FILE.md] [--trace-dir DIR]

Shapes:
  DM_rep4's imputation outputs: n = 4 301 held-out rows, 85 596 and 34 861 columns (the shared-memory regime, n <= 26 624);
  a tall one, 200 000 x 2 000 (20 % of a 10^6-cell run: the sort runs through global scratch), once with 5 % and once
  with 50 % positives (the sort's share of the time grows with the number of positives).
Scores are random fp32 (the timing does not depend on their values); measured is a scipy.sparse CSR matrix with 5 % of
its entries positive, as an AnnData .X would be, or a dense fp32 0 / 1 matrix at 50 %. For each shape: the host's positive lists (CSC of measured), the C call
alone, the whole imputation_auroc call (medians of 3 after a warm-up; every call ends in a synchronise), the device time
of its phases from a torch.profiler run (host-to-device copies, key transpose, per-column sort and search), and the
sklearn loop timed on a few columns and extrapolated to all of them. Agreement: the largest |difference| on those columns.
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


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def median_time(fn, reps=3):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out


def phases(fn, trace_dir, tag):
    """Device time per phase (ms) from one profiled call, by kernel / copy name."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    if trace_dir:
        prof.export_chrome_trace(os.path.join(trace_dir, 'auroc_' + ''.join(ch if ch.isalnum() else '_' for ch in tag) + '.json'))
    out = {}
    for ev in prof.key_averages():
        us = getattr(ev, 'device_time_total', None)
        if us is None:
            us = ev.cuda_time_total
        name = ev.key
        if 'k_auroc_keys' in name:
            ph = 'keys + transpose (k_auroc_keys)'
        elif 'k_auroc_col' in name:
            ph = 'sort + search (k_auroc_col)'
        elif 'HtoD' in name:
            ph = 'host-to-device copies'
        elif 'DtoH' in name:
            ph = 'device-to-host copies'
        else:
            ph = 'other (' + name[:40] + ')'
        if us > 0:
            out[ph] = out.get(ph, 0.0) + us / 1e3
    return out


def run(name, n, d, n_loop, density, trace_dir, seed=0):
    import scipy.sparse as sp
    from sklearn.metrics import roc_auc_score
    from jamie_b200 import _lib, evaluation
    rng = np.random.default_rng(seed)
    S = rng.standard_normal((n, d), dtype=np.float32)
    if density <= 0.05:
        M = sp.random(n, d, density=density, format='csr', dtype=np.float32, random_state=seed + 1)
        M.data += 0.1                                                    # every stored entry is a positive
    else:
        M = (rng.random((n, d), dtype=np.float32) < density).astype(np.float32)
    t_labels, (ptr, rows) = median_time(lambda: evaluation.positive_lists(M, 0.0, evaluation.BATCH_BYTES))

    u2, n_pos = np.empty(d, np.uint64), np.empty(d, np.int64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    lib = _lib.load()
    t_call, _ = median_time(lambda: _lib.check(lib.jb_metric_feature_auroc(p(S), n, d, p(ptr), p(rows), evaluation.BATCH_BYTES,
                                                                            0, p(u2), p(n_pos))))
    wall, got = median_time(lambda: evaluation.imputation_auroc(S, M, device=0))
    ph = phases(lambda: evaluation.imputation_auroc(S, M, device=0), trace_dir, name)

    cols = np.linspace(0, d - 1, n_loop).astype(int)
    Mc = M.tocsc() if sp.issparse(M) else M
    y = [(Mc[:, j].toarray() if sp.issparse(Mc) else Mc[:, j]).ravel() > 0 for j in cols]
    roc_auc_score(y[0], S[:, cols[0]])                                   # warm-up
    t0 = time.perf_counter()
    want = np.array([roc_auc_score(y[q], S[:, j]) for q, j in enumerate(cols)])
    t_loop = time.perf_counter() - t0
    return dict(name=name, n=n, d=d, measured=f"{'CSR' if sp.issparse(M) else 'dense'}, {density:.0%} positives", batches=-(-d // max(1, evaluation.BATCH_BYTES // ((16 if n <= 26624 else 24) * n))),
                labels_s=t_labels, call_s=t_call, wall_s=wall, phases_ms=ph, loop_cols=n_loop, loop_s=t_loop,
                loop_extrapolated_s=t_loop / n_loop * d, max_abs_diff=float(np.abs(got[cols] - want).max()),
                score_gb=4.0 * n * d / 1e9)


def report(rows, gpu, out):
    lines = ['# Per-feature AUROC: `imputation_auroc` against the `roc_auc_score` loop', '',
             f'Measured on: {gpu} (name, power limit), `python tools/auroc_bench.py`. Scores random fp32, threshold 0.', '']
    for r in rows:
        lines += [f"## {r['name']}: n = {r['n']}, d = {r['d']} ({r['score_gb']:.2f} GB of fp32 scores, "
                  f"{r['batches']} column batch(es) at the default BATCH_BYTES)", '',
                  f"- measured: {r['measured']}; positive lists on the host: {r['labels_s'] * 1e3:.1f} ms",
                  f"- `jb_metric_feature_auroc` call alone (lists given): {r['call_s'] * 1e3:.1f} ms "
                  f"({r['score_gb'] / r['call_s']:.1f} GB/s of scores)",
                  f"- `imputation_auroc` wall time (median of 3 after a warm-up, ends in a synchronise): "
                  f"{r['wall_s'] * 1e3:.1f} ms",
                  '- device time by phase (one profiled call; the copies run on their own stream and overlap the '
                  'previous batch\'s kernels):']
        for ph, ms in sorted(r['phases_ms'].items(), key=lambda kv: -kv[1]):
            lines.append(f'  - {ph}: {ms:.2f} ms')
        lines += [f"- `roc_auc_score` loop: {r['loop_s']:.2f} s for {r['loop_cols']} columns; extrapolated (not run) to all "
                  f"{r['d']} columns: {r['loop_extrapolated_s']:.0f} s ({r['loop_extrapolated_s'] / r['wall_s']:.0f}x the "
                  f"GPU call)",
                  f"- agreement on those columns: max |AUROC difference| {r['max_abs_diff']:.2e}", '']
    text = '\n'.join(lines)
    print(text)
    if out:
        with open(out, 'w') as f:
            f.write(text + '\n')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--quick', action='store_true', help='small shapes (a rehearsal)')
    ap.add_argument('--out', default=None)
    ap.add_argument('--trace-dir', default=None)
    a = ap.parse_args()
    import torch
    torch.cuda.set_device(0)
    gpu = card()
    if a.trace_dir:
        os.makedirs(a.trace_dir, exist_ok=True)
    if a.quick:
        shapes = [('held-out', 4301, 2000, 10, 0.05), ('tall', 30000, 50, 5, 0.5)]
    else:
        shapes = [('DM_rep4, 85 596 outputs', 4301, 85596, 40, 0.05), ('DM_rep4, 34 861 outputs', 4301, 34861, 40, 0.05),
                  ('tall', 200000, 2000, 10, 0.05), ('tall, half positive', 200000, 2000, 10, 0.5)]
    rows = [run(*s, trace_dir=a.trace_dir) for s in shapes]
    report(rows, gpu, a.out)


if __name__ == '__main__':
    main()
