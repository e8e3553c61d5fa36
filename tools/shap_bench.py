"""Shapley values (JAMIE.shap_values, jb_shapley) against the estimator run one masked batch at a time.

  python tools/shap_bench.py [--quick] [--out FILE.md] [--trace-dir DIR]

Shapes (SURVEY.md 3.2):
  dense : scMNC-Visual.ipynb -- n = 3 654, raw 1 302 -> 39, pca_dim [512, 512] (39 on the ephys side), latent 32;
          256 cells explained against 100 background rows, n_permutations = 2, all 39 outputs;
  sparse: DM_rep4 -- n = 4 301, raw 85 596 (about 10 % nonzero) -> 34 861, PCA 512 / 512, latent 32; 16 cells against
          100 background rows, n_permutations = 2, 50 selected outputs.
The models have random weights and synthetic PCA maps (timing does not depend on the values); only the explained and
background rows are generated. For each shape: the wall time of shap_values (median of 3 after one warm-up), the device
time of its phases from a torch.profiler run, chain rows per second and the steps skipped as inactive, and
naive_shap_values (modal_predict of every masked batch) timed on part of the work and extrapolated.
"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import impact_bench as IB  # noqa: E402  (make_jamie, card, median_time; puts the repository root on sys.path)
from jamie_b200.shapley import DeviceShapley  # noqa: E402


class Recording(DeviceShapley):
    """DeviceShapley that keeps the chain-row statistics {chain rows, skipped steps} of the last call."""
    stats = None

    def run(self, *a):
        super().run(*a)
        Recording.stats = a[12]


def phases(fn, trace_dir, tag):
    """Device time per phase (ms) from one profiled call, by kernel name."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    if trace_dir:
        prof.export_chrome_trace(os.path.join(trace_dir, f'shap_{tag}.json'))
    out = {}
    for ev in prof.key_averages():
        name = ev.key
        us = getattr(ev, 'device_time_total', None)
        if us is None:
            us = ev.cuda_time_total
        if 'k_shap_walk' in name or 'k_shap_chunk_start' in name or 'k_shap_count' in name:
            ph = 'walk build'
        elif 'persistent' in name or 'k_fold' in name or 'k_to_half' in name:
            ph = 'chain'
        elif 'k_split_tf32' in name or 'gemm_tf32_grouped' in name:
            ph = 'inverse GEMM'
        elif 'k_shap_fold' in name or 'k_shap_base' in name or 'k_shap_rows_f32' in name:
            ph = 'difference fold'
        else:
            ph = 'other (' + name[:40] + ')'
        if us > 0:
            out[ph] = out.get(ph, 0.0) + us / 1e3
    return out


def rows_of(rng, m, d, density):
    if density >= 1.0:
        return rng.standard_normal((m, d)) + rng.standard_normal(d)
    import scipy.sparse as sp
    A = sp.random(m, d, density=density, format='csr', random_state=np.random.RandomState(int(rng.integers(1 << 30))),
                  data_rvs=lambda k: rng.gamma(2.0, 1.0, k))
    return A


def run(name, n, d_raw, k, L, nx, nb, outputs, density, naive_chunks, trace_dir, seed=0):
    from jamie_b200 import shapley
    jm = IB.make_jamie(n, d_raw, k, L, seed)
    rng = np.random.default_rng(seed + 1)
    X = rows_of(rng, nx, d_raw[0], density)
    B = rows_of(rng, nb, d_raw[0], density)
    O = np.arange(d_raw[1]) if outputs is None else np.sort(rng.choice(d_raw[1], outputs, replace=False))
    call = lambda: shapley.shap_values(jm, X, 0, B, outputs=O, n_permutations=2, seed=seed, device=Recording)  # noqa: E731
    wall, res = IB.median_time(call)
    chain_rows, skipped = (int(v) for v in Recording.stats)
    ph = phases(call, trace_dir, name)
    # the naive estimator: modal_predict of every masked batch (WALK_ROWS rows of one walk, every step evaluated)
    predict = lambda A: np.asarray(jm.modal_predict(A, 0), np.float64)[:, O]   # noqa: E731
    d = d_raw[0]
    walks = 2 * nb                                   # per explained cell
    per_walk = -(-d // shapley.WALK_ROWS)
    x0 = shapley._dense(X[:1])[0]
    Bd = shapley._dense(B)
    perms = shapley.draw_permutations(d, 2, seed)
    if naive_chunks is None:                         # the whole estimator for one cell
        t0 = time.perf_counter()
        values, _ = shapley.naive_shap_values(predict, x0[None], Bd, perms)
        t_naive = time.perf_counter() - t0
        naive = dict(what='1 cell, run in full', run_s=t_naive, per_cell_s=t_naive,
                     norm_rel=float(np.linalg.norm(res.values[0] - values[0]) / np.linalg.norm(values[0])))
    else:                                            # a few masked batches of one walk, as _naive_sums builds them
        rank = np.empty(d, np.int64)
        rank[perms[0]] = np.arange(d)
        predict(Bd[:2])
        t0 = time.perf_counter()
        for c in range(naive_chunks):
            t = np.arange(c * shapley.WALK_ROWS, min(d, (c + 1) * shapley.WALK_ROWS))
            predict(np.where(rank[None, :] <= t[:, None], x0[None, :], Bd[0][None, :]))
        t_naive = time.perf_counter() - t0
        naive = dict(what=f'{naive_chunks} masked batches of {shapley.WALK_ROWS} rows timed', run_s=t_naive,
                     per_cell_s=t_naive / naive_chunks * walks * per_walk)
    naive['all_cells_s'] = naive['per_cell_s'] * nx
    jm.engine.close()
    return dict(name=name, n=n, d_raw=d_raw, k=k, L=L, nx=nx, nb=nb, n_out=len(O), density=density, wall_s=wall,
                phases_ms=ph, chain_rows=chain_rows, skipped=skipped, naive=naive)


def report(rows, gpu, out):
    lines = ['# Shapley values: `JAMIE.shap_values` against the estimator run one masked batch at a time', '',
             f'Measured on: {gpu} (name, power limit), `python tools/shap_bench.py`.', '']
    for r in rows:
        dens = 'dense' if r['density'] >= 1 else f"{r['density'] * 100:.0f} % nonzero"
        lines += [f"## {r['name']}: n = {r['n']}, raw {r['d_raw'][0]} ({dens}) -> {r['d_raw'][1]}, PCA {r['k'][0]} / "
                  f"{r['k'][1]}, latent {r['L']}; {r['nx']} cells x {r['nb']} background rows, 2 permutations, "
                  f"{r['n_out']} outputs", '',
                  f"- `shap_values` wall time (median of 3 after a warm-up): {r['wall_s']:.3f} s",
                  f"- chain rows: {r['chain_rows']:,} ({r['chain_rows'] / r['wall_s'] / 1e6:.1f} M rows/s of wall time); "
                  f"steps skipped as inactive: {r['skipped']:,} "
                  f"({100.0 * r['skipped'] / max(1, r['skipped'] + r['chain_rows']):.1f} % of all walk steps)",
                  '- device time by phase (one profiled call):']
        for ph, ms in sorted(r['phases_ms'].items(), key=lambda kv: -kv[1]):
            lines.append(f'  - {ph}: {ms:.1f} ms')
        nv = r['naive']
        lines.append(f"- `naive_shap_values` (one `modal_predict` per masked batch): {nv['what']}: {nv['run_s']:.2f} s; "
                     f"extrapolated (not run): {nv['per_cell_s']:.1f} s per cell, {nv['all_cells_s']:.0f} s for all "
                     f"{r['nx']} cells ({nv['all_cells_s'] / r['wall_s']:.0f}x the batched call)")
        if 'norm_rel' in nv:
            lines.append(f"- agreement with it on that cell: relative norm difference {nv['norm_rel']:.2e}")
        lines.append('')
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
    gpu = IB.card()
    if a.trace_dir:
        os.makedirs(a.trace_dir, exist_ok=True)
    if a.quick:
        shapes = [('dense', 300, (130, 39), (64, 39), 16, 8, 10, None, 1.0, None),
                  ('sparse', 300, (9000, 700), (64, 48), 16, 2, 10, 50, 0.1, 1)]
    else:
        shapes = [('dense', 3654, (1302, 39), (512, 39), 32, 256, 100, None, 1.0, None),
                  ('sparse', 4301, (85596, 34861), (512, 512), 32, 16, 100, 50, 0.1, 2)]
    rows = [run(*s, trace_dir=a.trace_dir) for s in shapes]
    report(rows, gpu, a.out)


if __name__ == '__main__':
    main()
