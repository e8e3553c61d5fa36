"""Feature ablation (JAMIE.feature_impact, jb_feature_impact) against the per-feature loop it replaces.

  python tools/impact_bench.py [--quick] [--out FILE.md] [--trace-dir DIR]

Shapes (SURVEY.md 3.2):
  imputation: DM_rep4-Imp.ipynb -- n = 4 301, raw widths 85 596 -> 34 861, PCA 512 on both sides, latent 32, 464 features,
              with a target;
  latent    : brainchromatin.ipynb's scan -- n = 500, raw width 19 836 with PCA 512, space='latent', all 19 836 features.
The models have random weights and synthetic PCA maps (timing does not depend on the values). For each shape: the wall
time of feature_impact (median of 3 after one warm-up), the device time of its phases from a torch.profiler run (input
build k_ablate_rows, the folded chain, the inverse GEMM with its split, the moments), the TF32 rate of the inverse GEMM,
and the loop (modal_predict / transform_one of every ablated matrix + imputation_correlation) timed on a few features and
extrapolated to all of them. Agreement: the largest |difference| of r (or of shift) on those features.
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

TF32_PEAK = 1125e12   # HGX B200 data sheet, one GPU, dense TF32


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def make_jamie(n, d_raw, k, L, seed):
    """A JAMIE with random weights and linear PCA maps [k_i, d_i] on both sides, attached to a fresh engine."""
    import torch
    from sklearn.decomposition import PCA
    from jamie_b200.jamie import JAMIE
    from jamie_b200.model import edModelVar
    from jamie_b200.utilities import preclass
    rng = np.random.default_rng(seed)
    pres = []
    for i in range(2):
        pca = PCA(k[i])
        pca.components_ = (rng.standard_normal((k[i], d_raw[i]), dtype=np.float32) / np.sqrt(d_raw[i])).astype(np.float32)
        pca.mean_ = rng.standard_normal(d_raw[i], dtype=np.float32)
        sample = rng.standard_normal((n, k[i])) * np.linspace(3, 0.1, k[i])
        pres.append(preclass(sample, pca=pca))
    torch.manual_seed(seed)
    jm = JAMIE(output_dim=L)
    jm.model = edModelVar(list(k), L, preprocessing=[p.transform for p in pres],
                          preprocessing_inverse=[p.inverse_transform for p in pres])
    jm.dataset_num = 2
    jm.model.eval()
    jm._ensure_engine()
    return jm


def median_time(fn, reps=3):
    import torch
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out


def phases(fn, trace_dir, tag):
    """Device time per phase (ms) from one profiled call, by kernel name."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    if trace_dir:
        prof.export_chrome_trace(os.path.join(trace_dir, f'impact_{tag}.json'))
    out = {}
    for ev in prof.key_averages():
        name = ev.key
        us = getattr(ev, 'device_time_total', None)
        if us is None:
            us = ev.cuda_time_total
        if 'k_ablate_rows' in name:
            ph = 'input build'
        elif 'persistent' in name or 'k_fold' in name or 'k_to_half' in name:
            ph = 'chain'
        elif 'k_split_tf32' in name or 'gemm_tf32_grouped' in name:
            ph = 'inverse GEMM'
        elif 'k_impact_moments' in name:
            ph = 'moments'
        else:
            ph = 'other (' + name[:40] + ')'
        if us > 0:
            out[ph] = out.get(ph, 0.0) + us / 1e3
    gemm_ms = sum(ev.device_time_total if hasattr(ev, 'device_time_total') else ev.cuda_time_total
                  for ev in prof.key_averages() if 'gemm_tf32_grouped' in ev.key) / 1e3
    return out, gemm_ms


def run(name, n, d_raw, k, L, F, space, n_loop, trace_dir, seed=0):
    from jamie_b200.evaluation import imputation_correlation
    from jamie_b200.impact import naive_feature_impact
    jm = make_jamie(n, d_raw, k, L, seed)
    rng = np.random.default_rng(seed + 1)
    X = rng.standard_normal((n, d_raw[0]), dtype=np.float32) + rng.standard_normal(d_raw[0], dtype=np.float32)
    T = rng.standard_normal((n, d_raw[1]), dtype=np.float32) if space == 'output' else None
    J = np.arange(F)
    call = lambda: jm.feature_impact(X, 0, target=T, features=J, space=space)   # noqa: E731
    wall, res = median_time(call)
    ph, gemm_ms = phases(call, trace_dir, name)
    # the loop on the first n_loop features (plus its baseline prediction), extrapolated to F
    predict = (lambda A: jm.modal_predict(A, 0)) if space == 'output' else (lambda A: jm.transform_one(A, 0))
    fills = X[:, :n_loop].astype(np.float64).mean(0)
    naive_feature_impact(predict, X, J[:1], fills[:1], T, pearson=imputation_correlation)   # warm-up
    t0 = time.perf_counter()
    shift, base_r, r = naive_feature_impact(predict, X, J[:n_loop], fills, T, pearson=imputation_correlation)
    t_loop = time.perf_counter() - t0
    per_feature = t_loop / (n_loop + 1)
    agree = {'shift_max_abs': float(np.abs(res.shift[:n_loop] - shift).max()),
             'shift_norm_rel': float(np.linalg.norm(res.shift[:n_loop] - shift) / np.linalg.norm(shift))}
    if T is not None:
        agree['r_max_abs'] = float(np.nanmax(np.abs(res.r[:n_loop] - r)))
        agree['baseline_r_max_abs'] = float(np.nanmax(np.abs(res.baseline_r - base_r)))
    flops = 2.0 * n * F * k[1] * d_raw[1] if space == 'output' else 0.0   # useful products of the ablated rows
    jm.engine.close()
    return dict(name=name, n=n, d_raw=d_raw, k=k, L=L, F=F, space=space, wall_s=wall, phases_ms=ph, gemm_ms=gemm_ms,
                gemm_useful_tflops=flops / (gemm_ms / 1e3) / 1e12 if gemm_ms else None,
                gemm_tf32_tflops=3 * flops / (gemm_ms / 1e3) / 1e12 if gemm_ms else None,
                loop_features=n_loop, loop_s=t_loop, loop_extrapolated_s=per_feature * (F + 1), agreement=agree)


def report(rows, gpu, out):
    lines = [f'# Feature ablation: `JAMIE.feature_impact` against the per-feature loop', '',
             f'Measured on: {gpu} (name, power limit), `python tools/impact_bench.py`.', '']
    for r in rows:
        lines += [f"## {r['name']}: n = {r['n']}, raw {r['d_raw'][0]} -> {r['d_raw'][1]}, PCA {r['k'][0]} / {r['k'][1]}, "
                  f"latent {r['L']}, {r['F']} features, space = '{r['space']}'", '',
                  f"- `feature_impact` wall time (median of 3 after a warm-up): {r['wall_s']:.3f} s",
                  '- device time by phase (one profiled call):']
        for ph, ms in sorted(r['phases_ms'].items(), key=lambda kv: -kv[1]):
            lines.append(f'  - {ph}: {ms:.1f} ms')
        if r['gemm_tf32_tflops']:
            lines.append(f"- inverse GEMM (3xTF32): {r['gemm_ms']:.1f} ms; {r['gemm_useful_tflops']:.0f} TFLOP/s of fp32 products "
                         f"(2 n F k d_out, ablated rows only), {r['gemm_tf32_tflops']:.0f} TFLOP/s of TF32 tensor work (3x), "
                         f"against the data sheet's {TF32_PEAK / 1e12:.0f} TFLOP/s dense TF32")
        lines += [f"- loop: {r['loop_s']:.2f} s for {r['loop_features']} features plus the baseline prediction; "
                  f"extrapolated (not run) to all {r['F']} features: {r['loop_extrapolated_s']:.0f} s "
                  f"({r['loop_extrapolated_s'] / r['wall_s']:.0f}x the batched call)",
                  f"- agreement on those features: " + ', '.join(f'{k} {v:.2e}' for k, v in r['agreement'].items()), '']
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
        shapes = [('imputation', 301, (900, 700), (64, 48), 16, 24, 'output', 3),
                  ('latent', 100, (500, 300), (64, 48), 16, 200, 'latent', 3)]
    else:
        shapes = [('imputation', 4301, (85596, 34861), (512, 512), 32, 464, 'output', 3),
                  ('latent', 500, (19836, 2000), (512, 512), 32, 19836, 'latent', 5)]
    rows = [run(*s, trace_dir=a.trace_dir) for s in shapes]
    report(rows, gpu, a.out)


if __name__ == '__main__':
    main()
