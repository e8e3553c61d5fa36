"""Where does a long run of the bench workload leave the finite range? Prints the loss trajectory and the first
non-finite step on the bench's own data, plan and seeds (N = 1)."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
import torch
import bench as Bn
from jamie_b200.engine import Engine

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 2200
n = int(sys.argv[2]) if len(sys.argv) > 2 else Bn.N_CELLS
torch.cuda.set_device(0)
g = torch.Generator(device='cuda').manual_seed(1234)
data = [torch.randn((n, d), generator=g, device='cuda', dtype=torch.float32) for d in Bn.DIMS]
SEEDS = [int(x) for x in os.environ.get('JB_DIV_SEEDS', '0').split(',')]
for seed in SEEDS:
    rng = np.random.default_rng(100 + seed)
    mask = (rng.random(n) < 0.5).astype(np.float32)
    nz = np.flatnonzero(mask)[:2]
    cs = np.stack([nz, nz], 1)
    params, bufs = Bn.init_params()
    eng = Engine(Bn.DIMS, Bn.LATENT, Bn.BATCH, Bn.DROPOUT, seed=666 * 1000003 + seed)
    eng.set_params(params); eng.set_bn_stats(bufs)
    for i in range(2):
        eng.set_dataset(i, data[i])
    eng.set_prior_diag(mask); eng.set_f_dense(None)
    idx0, idx1 = Bn.make_plan(n, steps, rng, cs)
    eng.upload_plan(idx0, idx1, np.full(steps, 0.5))
    eng.train_steps(steps)
    torch.cuda.synchronize()
    ls = eng.read_losses(steps)
    bad = np.flatnonzero(~np.isfinite(ls[:, :6]).all(axis=1))
    print(f'seed {seed}: max total loss {np.nanmax(ls[:, 4]):.3g} at step {int(np.nanargmax(ls[:, 4]))}, max |g| {np.nanmax(ls[:, 5]):.3g}; first non-finite step: {int(bad[0]) if bad.size else None} of {steps}')
    for s in (list(range(0, steps, max(steps // 16, 1))) if os.environ.get('JB_DIV_VERBOSE') else []) + ([int(bad[0]) - 2, int(bad[0]) - 1, int(bad[0])] if bad.size else []):
        if 0 <= s < steps:
            print(f'  step {s:5d}: KL {ls[s, 0]:.4g} Rec {ls[s, 1]:.4g} Cos {ls[s, 2]:.4g} F {ls[s, 3]:.4g} total {ls[s, 4]:.4g} |g| {ls[s, 5]:.4g}')
    if bad.size and os.environ.get('JB_DIV_DUMP'):
        # replay up to the step before the first non-finite one (runs are bit-reproducible), then that step alone: which taps
        # leave the finite range first?
        s0 = int(bad[0])
        eng.close()
        eng = Engine(Bn.DIMS, Bn.LATENT, Bn.BATCH, Bn.DROPOUT, seed=666 * 1000003 + seed)
        eng.set_params(params); eng.set_bn_stats(bufs)
        for i in range(2):
            eng.set_dataset(i, data[i])
        eng.set_prior_diag(mask); eng.set_f_dense(None)
        eng.upload_plan(idx0, idx1, np.full(steps, 0.5))
        if s0 > 0:
            eng.train_steps(s0)
        th = eng.debug_read('theta', (1, 1 << 26)).ravel()
        print(f'  before step {s0}: theta finite {np.isfinite(th).all()}, max |theta| {np.abs(th).max():.4g}')
        eng.train_steps(1)
        torch.cuda.synchronize()
        B, L, D = Bn.BATCH, Bn.LATENT, Bn.DIMS
        shapes = {'mulv': [2 * L] * 2, 'z': [L] * 2, 'c': [L] * 2, 'g1_': D, 'g2_': [2 * d for d in D], 'xhat': D, 'dxhat': D, 'dg2_': [2 * d for d in D],
                  'dy4_': [2 * d for d in D], 'dg1_': D, 'dy3_': D, 'dc': [L] * 2, 'dmulv': [2 * L] * 2, 'dh2_': D, 'dy2_': D, 'dh1_': [2 * d for d in D],
                  'dy1_': [2 * d for d in D]}
        for key, w in shapes.items():
            for i in range(2):
                t = eng.debug_read(f'{key}{i}', (B, w[i]))
                fin = np.isfinite(t)
                rows = np.flatnonzero(~fin.all(axis=1))
                print(f'  {key}{i}: non-finite {int((~fin).sum())} of {t.size} (rows {rows[:6].tolist()}), finite max {np.abs(np.where(fin, t, 0)).max():.4g}')
        gr = eng.debug_read('grad', (1, 1 << 26)).ravel()
        print(f'  grad: non-finite {int((~np.isfinite(gr)).sum())} of {gr.size}')
    eng.close()
