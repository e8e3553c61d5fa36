"""Benchmark of the JAMIE hot path on B200: train cells/sec (fwd + bwd + clip + Adam) of the coupled VAE.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (BASELINE.json configs[3], the configuration the metric is quoted on, at EVERY N): synthetic 1M-cell pair,
post-PCA widths [512, 512], output_dim 32, batch 512 per rank, 50 % partially matched P (diag mask -> 'hybrid' sampler),
dropout 0.6, F = 0; the cells are sharded over the ranks (weak scaling: per-rank batch fixed), one all-reduce of the flat
gradient buffer per step for N > 1. Data are synthetic standardised fp32 rows of the named shape; weights are the
reference's random init (torch seed 666). A "step" is one optimizer step over one batch.

  value : cells/s, whole job, data and sampling plan resident in HBM; the K steps are ONE launch of the persistent step
          kernel (N = 1) timed with CUDA events
  e2e   : cells/s through the C ABI with HOST data: per step the batch is gathered on the host into pinned memory,
          copied to the device inside jb_hostbatch_submit, and the loss scalars are read back
  e2e_fit_transform : wall clock of the user-facing call, JAMIE(...).fit_transform on host numpy arrays (standardise,
          upload, sampler, training chunks, loss read-back, final encode, download)
  roofline      : the step kernel (k_step: the whole step is one kernel) against the measured HBM peak with the
          compulsory bytes of a step (fp32 param + Adam moments r/w + gathered inputs, SURVEY.md 8d); DRAM traffic from
          the committed `ncu --set full` capture
  gemm_roofline : all GEMM phases together (algorithmic FLOPs / in-kernel phase time) against the measured tensor peak
  step_profile  : microseconds per phase INSIDE the persistent kernel (GPU global timer at the phase boundaries)
  cpu_baseline  : the reference itself (oracle/_ref = a copy of /root/reference/jamie made by build()) timed on this
          box's host cores; falls back to the numpy oracle port when the copy is absent
`--impl reference` times the reference alone (all host cores; rank 0 only under torchrun).
`--dump-outputs DIR` writes what the last timed step left to its caller as DIR/<name>.npy (see dump_outputs); the inputs
depend on the arguments only, so two builds can be compared output for output.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DIMS, LATENT, BATCH, DROPOUT = [512, 512], 32, 512, 0.6
N_CELLS = 1_000_000
N_PARAMS = 4312194
ALG_BYTES_PER_STEP = 6 * 4 * N_PARAMS + 4 * BATCH * sum(DIMS)      # SURVEY.md 8d: 105.6 MB
ALG_FLOPS_PER_STEP = 12.11e9


def load_peaks():
    try:
        pk = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        return {'hbm_gbs': pk['hbm_gbs'], 'bf16_tflops': pk['bf16_tflops'],
                'bf16_tflops_sustained': pk.get('bf16_tflops_sustained', pk['bf16_tflops']), 'source': 'measured'}
    except Exception:
        return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback'}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for k, nm in enumerate(names):
                    if r[3 + k].lower().startswith('active'):
                        reasons.add(nm)
            except Exception:
                pass
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx or None, 'reasons': sorted(reasons),
                'samples': len(sm)}


def make_plan(n, steps, rng, corr_samples):
    """The reference's 'hybrid' sampler (jamie/jamie.py:559-573) for a partially matched diagonal prior."""
    idx0 = np.empty((steps, BATCH), np.int64)
    idx1 = np.empty((steps, BATCH), np.int64)
    for s in range(steps):
        k = min(int(np.sum(rng.random(BATCH) < .8)), 2)
        ci = rng.choice(2, k, replace=False)
        idx0[s] = np.concatenate([corr_samples[0][ci], rng.choice(n, BATCH - k, replace=False)])
        idx1[s] = np.concatenate([corr_samples[1][ci], rng.choice(n, BATCH - k, replace=False)])
    return idx0, idx1


def init_params():
    import torch
    from jamie_b200.model import edModelVar
    torch.manual_seed(666)
    m = edModelVar(DIMS, LATENT, dropout=DROPOUT)
    return m.packed_parameters(), m.packed_buffers()


# ------------------------------------------------------------------------------------------------ CPU arms
def cpu_reference(steps, warmup, n=4096):
    """The UNMODIFIED reference (oracle/_ref, or /root/reference in the build container) on this box's host cores, timed
    as BASELINE.md section 3 prescribes: its own project_jamie loop on synthetic data of the benchmark's shape with n
    capped (its per-step cost does not depend on n, its set-up is O(n^2)), use_f_tilde=False, and the per-batch laps of its
    own time_logger ('Get subset samples' ... 'Step') summed over `steps` optimizer steps after `warmup`."""
    import torch
    from oracle import ref_harness as RH
    torch.set_num_threads(os.cpu_count() or 1)
    jamie = RH.import_reference()
    import jamie.jamie as JJ
    loggers = []
    base = JJ.time_logger

    class Spy(base):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            loggers.append(self)

    JJ.time_logger = Spy
    rng = np.random.default_rng(0)
    data = [rng.standard_normal((n, d)) for d in DIMS]
    m = (rng.random(n) < 0.5).astype(np.float64)
    per_epoch = max(1, n // BATCH)
    epochs = -(-(steps + warmup) // per_epoch)
    np.random.seed(42)
    try:
        jm = jamie.JAMIE(output_dim=LATENT, batch_size=BATCH, pca_dim=None, dropout=DROPOUT, use_f_tilde=False,
                         epoch_DNN=epochs, min_epochs=10 * epochs, log_DNN=10 ** 9, use_early_stop=False)
        with contextlib.redirect_stdout(io.StringIO()):
            jm.fit_transform(dataset=data, P=np.diag(m))
    finally:
        JJ.time_logger = base
    hist = max((lg.history for lg in loggers), key=lambda h: len(h.get('Step', [])))
    labels = [k for k in hist if k not in ('Setup', 'Output')]
    w, k = warmup, steps
    if len(hist['Step']) < w + k:
        raise RuntimeError(f'the reference ran {len(hist["Step"])} optimizer steps, {w + k} were asked for')
    total = sum(float(np.sum(hist[lb][w:w + k])) for lb in labels if len(hist[lb]) >= w + k)
    return {'value': BATCH * k / total, 'unit': 'cells/s', 'cores': os.cpu_count(), 'kind': 'reference',
            'threads': torch.get_num_threads(), 'ms_per_step': 1e3 * total / k, 'steps': k, 'warmup': w,
            'sample': f'{k} optimizer steps (after {w} warm-up) of the reference\'s own project_jamie loop, batch {BATCH}, widths '
                      f'{DIMS}, output_dim {LATENT}, dropout {DROPOUT}, n = {n} cells, torch {torch.__version__} CPU; sum of '
                      f'its time_logger laps {labels}, {total:.1f} s'}


def cpu_port(steps, warmup):
    """Fallback when the reference copy is absent: the numpy oracle port of one reference optimizer step, timed over
    `steps` steps after `warmup`."""
    from oracle import jamie_oracle as O
    rng = np.random.default_rng(0)
    n = 8192
    data = [rng.standard_normal((n, d)).astype(np.float32) for d in DIMS]
    m = (rng.random(n) < 0.5).astype(np.float32)
    nz = np.flatnonzero(m)[:2]
    params, _ = init_params()
    orc = O.OracleModel(DIMS, LATENT, dropout=DROPOUT, params=params)
    cs = np.stack([nz, nz], 1)

    def one(step):
        i0, i1 = make_plan(n, 1, rng, cs)
        i0, i1 = i0[0], i1[0]
        x = [data[0][i0], data[1][i1]]
        Pb = (i0[:, None] == i1[None, :]).astype(np.float32) * m[i0][:, None]
        s = Pb.sum(1)
        s[s == 0] = 1
        corr = Pb / s[:, None]
        eps = [rng.standard_normal((BATCH, LATENT)).astype(np.float32) for _ in range(2)]
        widths = [1024, 512, 1024, 512, 512, 1024, 512, 1024]
        masks = [(rng.random((BATCH, w)) >= DROPOUT).astype(np.uint8) for w in widths]
        orc.train_step(x, corr, np.zeros((BATCH, BATCH), np.float32), eps, masks, 0.5)

    for s in range(warmup):
        one(s)
    t0 = time.perf_counter()
    for s in range(steps):
        one(s)
    dt = time.perf_counter() - t0
    return {'value': BATCH * steps / dt, 'unit': 'cells/s', 'cores': os.cpu_count(), 'kind': 'port',
            'sample': f'{steps} optimizer steps (after {warmup} warm-up) of batch {BATCH} at widths {DIMS}, output_dim {LATENT} '
                      f'(numpy fp32 oracle, BLAS on all host cores), {dt:.1f} s', 'ms_per_step': 1e3 * dt / steps,
            'steps': steps, 'warmup': warmup}


def cpu_baseline(steps=60, warmup=10):
    from oracle import ref_harness as RH
    if RH.reference_available():
        try:
            return cpu_reference(steps, warmup)
        except Exception as ex:   # a broken copy must not take the GPU numbers down with it
            cb = cpu_port(steps, warmup)
            cb['note'] = f'reference copy failed to run ({type(ex).__name__}: {ex}); oracle port timed instead'
            return cb
    return cpu_port(steps, warmup)


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    cb = cpu_baseline(steps=args.steps, warmup=args.warmup)
    line = {
        'impl': 'reference', 'metric': 'train cells/sec (fwd+bwd+Adam)', 'value': cb['value'], 'unit': 'cells/s',
        'n_gpus': args.gpus, 'steps': cb['steps'], 'warmup': cb['warmup'], 'ms_per_step': cb['ms_per_step'],
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args.gpus),
        'cpu_baseline': cb,
        'e2e': {'value': cb['value'], 'unit': 'cells/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def ncu_traffic(kernel_key):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/), or None."""
    try:
        t = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')))
        return t.get(kernel_key)
    except Exception:
        return None


def predict_leg(eng, torch, peaks, stream, rows_dev=1_250_000, rows_host=1 << 18):
    """modal_predict (BASELINE metric 2, configs[4]: 10M cells over 8 GPUs = 1.25M rows per rank): modality 0 -> 1 on
    pre-transformed [N, 512] fp32 rows. value: rows resident in HBM, CUDA events; e2e: pinned host buffers in and out
    through jb_predict."""
    g = torch.Generator(device='cuda').manual_seed(2)
    x = torch.randn((rows_dev, DIMS[0]), generator=g, device='cuda', dtype=torch.float32)
    out = torch.empty((rows_dev, DIMS[1]), device='cuda', dtype=torch.float32)
    l0 = eng.launch_count()
    eng.predict_into(0, 1, x.data_ptr(), 1 << 16, DIMS[0], out.data_ptr(), DIMS[1], 1, stream)   # warm-up, folds BN
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.predict_into(0, 1, x.data_ptr(), rows_dev, DIMS[0], out.data_ptr(), DIMS[1], 1, stream)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    assert bool(torch.isfinite(out[::4097]).all())
    del x, out
    hx = torch.randn((rows_host, DIMS[0]), dtype=torch.float32).pin_memory()
    ho = torch.empty((rows_host, DIMS[1]), dtype=torch.float32).pin_memory()
    eng.predict_into(0, 1, hx.data_ptr(), rows_host, DIMS[0], ho.data_ptr(), DIMS[1], 0, stream)
    t0 = time.perf_counter()
    eng.predict_into(0, 1, hx.data_ptr(), rows_host, DIMS[0], ho.data_ptr(), DIMS[1], 0, stream)
    dt = time.perf_counter() - t0
    flops_row = 2.0 * (2 * DIMS[0] * DIMS[0] * 2 + DIMS[0] * LATENT + LATENT * DIMS[1] + 2 * DIMS[1] * DIMS[1] * 2)
    v = rows_dev / (ms * 1e-3)
    return {'metric': 'modal_predict cells/sec', 'value': v, 'unit': 'cells/s', 'rows': rows_dev, 'ms': ms,
            'e2e': {'value': rows_host / dt, 'unit': 'cells/s', 'rows': rows_host,
                    'h2d_bytes': rows_host * DIMS[0] * 4, 'd2h_bytes': rows_host * DIMS[1] * 4},
            'roofline': {'bound': 'tensor', 'achieved': v * flops_row / 1e12, 'peak': peaks['bf16_tflops_sustained'],
                         'unit': 'TFLOP/s', 'frac': v * flops_row / 1e12 / peaks['bf16_tflops_sustained'],
                         'flops_per_row': flops_row},
            'gpu_launches': eng.launch_count() - l0}


def fit_transform_leg(torch, n=100_000, epochs=10):
    """Wall clock of the user-facing call: JAMIE(...).fit_transform(dataset=[X0, X1], P=mask) on host numpy arrays that
    already have the post-PCA width (pca_dim=None: per-feature standardisation only), then the embeddings come back as
    numpy. Everything a user waits for is inside: standardise, engine creation, upload, batch sampler, training chunks,
    loss read-back, final encode of all cells, download."""
    from jamie import JAMIE
    rng = np.random.default_rng(7)
    data = [rng.standard_normal((n, d)).astype(np.float32) for d in DIMS]
    mask = (rng.random(n) < 0.5).astype(np.float32)
    np.random.seed(0)
    out = {}
    for tag, ep in (('warm', 1), ('timed', epochs)):
        jm = JAMIE(output_dim=LATENT, batch_size=BATCH, pca_dim=None, dropout=DROPOUT, use_f_tilde=False, epoch_DNN=ep,
                   min_epochs=10 * ep, log_DNN=10 ** 9, use_early_stop=False)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            emb = jm.fit_transform(dataset=data, P=mask)
        dt = time.perf_counter() - t0
        steps = ep * (n // BATCH)
        out[tag] = (dt, steps)
        assert emb[0].shape == (n, LATENT) and np.all(np.isfinite(emb[0][::997]))
        jm.engine.close()
    dt, steps = out['timed']
    dt_w, steps_w = out['warm']
    per_step = (dt - dt_w) / max(1, steps - steps_w)
    return {'value': BATCH * steps / dt, 'unit': 'cells/s', 'seconds': dt, 'optimizer_steps': steps, 'cells': n, 'epochs': epochs,
            'marginal_us_per_step': 1e6 * per_step,
            'note': 'wall clock of JAMIE.fit_transform on host numpy data (pca_dim=None), incl. standardise, upload, sampler, '
                    'training, final encode, download; marginal_us_per_step = (T(10 epochs) - T(1 epoch)) / extra steps'}


def dump_outputs(eng, last_losses, out_dir):
    """The results of the last timed optimizer step, float32, packed in the reference's parameter / BatchNorm order:
    losses (KL, Rec, CosSim, F, total, pre-clip gradient norm), grads (that step's gradients), params and bn_stats
    (running mean, running var per BatchNorm layer) after its update. 34.5 MB at the benchmark's shape."""
    os.makedirs(out_dir, exist_ok=True)
    bn = eng.get_bn_stats()
    arrays = {
        'losses': np.asarray(last_losses[:6], np.float32),
        'grads': np.concatenate([g.ravel() for g in eng.get_grads()]),
        'params': eng.get_params(as_list=False),
        'bn_stats': np.concatenate([v for k, v in bn.items() if not k.endswith('.num_batches_tracked')]),
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def workload_config(n_gpus):
    wl = f'BASELINE configs[3]: synthetic 1M-cell pair sharded over {n_gpus} rank(s), widths [512,512], output_dim 32, ' \
         f'batch 512 per rank, 50% partially matched diagonal P (hybrid sampler), dropout 0.6, F=0' + \
         (', one flat-gradient all-reduce/step' if n_gpus > 1 else '')
    return {'workload': wl, 'cells': N_CELLS, 'widths': DIMS, 'output_dim': LATENT, 'batch_per_rank': BATCH,
            'parallelism': f'dp{n_gpus}', 'l2_policy': 'inputs larger than L2: every step gathers 2 x 512 random rows from a '
            '4.1 GB (N=1) resident dataset; parameters + Adam state (69 MB) are re-read every step by design'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=2000)
    ap.add_argument('--warmup', type=int, default=200)
    ap.add_argument('--impl', default='ours')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-predict', action='store_true')
    ap.add_argument('--no-fit', action='store_true')
    ap.add_argument('--predict-only', action='store_true', help='modal_predict leg alone (tuning runs)')
    ap.add_argument('--profile', action='store_true', help='device-resident steps only (for ncu): no e2e / stage / CPU legs, no JSON line')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the results of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and (args.impl == 'reference' or args.predict_only):
        ap.error('--dump-outputs writes the results of the timed training steps: not with --impl reference or --predict-only')
    if args.impl == 'reference':
        return run_reference(args)

    # stdout carries exactly one JSON line: anything libraries print on the way (e.g. NCCL's version banner) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(obj), flush=True)
        os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local)
    if world > 1:
        # 17 MB all-reduce per step: measured on 8 B200 375.7 us/step with NVLS off vs 392.5 us/step with NCCL's default
        os.environ.setdefault('NCCL_NVLS_ENABLE', '0')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    from jamie_b200.engine import Engine
    peaks = load_peaks()
    K, W = args.steps, max(args.warmup, 3)

    n = N_CELLS // world
    g = torch.Generator(device='cuda').manual_seed(1234 + rank)
    data = [torch.randn((n, d), generator=g, device='cuda', dtype=torch.float32) for d in DIMS]
    rng = np.random.default_rng(100 + rank)
    mask = (rng.random(n) < 0.5).astype(np.float32)
    nz = np.flatnonzero(mask)[:2]
    cs = np.stack([nz, nz], 1)
    params, bufs = init_params()
    eng = Engine(DIMS, LATENT, BATCH, DROPOUT, seed=666 * 1000003 + rank, device=local, world_size=world)
    eng.set_params(params)
    eng.set_bn_stats(bufs)
    stream = torch.cuda.current_stream().cuda_stream
    for i in range(2):
        eng.set_dataset(i, data[i], stream)
    eng.set_prior_diag(mask)
    eng.set_f_dense(None)
    idx0, idx1 = make_plan(n, W + K, rng, cs)
    eng.upload_plan(idx0, idx1, np.full(W + K, 0.5), stream)
    gx = None
    if world > 1:
        from jamie_b200.dp import GradExchange
        gx = GradExchange(eng)
        eng.upload_plan(idx0, idx1, np.full(W + K, 0.5), stream)   # (the step tables were rebuilt around the exchange buffer)
    if args.predict_only:
        p = predict_leg(eng, torch, peaks, stream)
        emit({k: p[k] for k in ('value', 'ms', 'e2e', 'gpu_launches')})
        eng.close()
        return

    def run_steps(k):
        if world == 1 or gx.mode == 'kernel':
            eng.train_steps(k, stream)          # ONE launch of the persistent step kernel for k optimizer steps (N > 1: the
                                                # kernel exchanges the gradients over peer memory itself)
        else:
            for _ in range(k):                  # backward | one all-reduce of the flat gradient buffer | update
                eng.step_backward(stream)
                gx.all_reduce()
                eng.step_update(stream)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident throughput
    run_steps(W)
    sync_all()
    l0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        e0.record()
        run_steps(K)
        e1.record()
        torch.cuda.synchronize()
    sync_all()
    ms = e0.elapsed_time(e1)
    launches = eng.launch_count() - l0
    if world > 1:
        t = torch.tensor([ms], device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    losses = eng.read_losses(W + K, stream)
    # The noise workload blows single latent rows up every few hundred steps (profiles/stability_r2.md). Such a step may
    # overflow the fp32 gradient NORM itself (|g| = inf; the reference's clip_grad_norm_ does the same) and is then a
    # zero update; the run is only valid if training carries on afterwards: the last tenth of the steps must be finite
    # and at most 1 % of all steps may show a non-finite scalar. The count is reported.
    finite_rows = np.isfinite(losses[:, :6]).all(axis=1)
    nonfinite_steps = int((~finite_rows).sum())
    assert finite_rows[-max(1, (W + K) // 10):].all() and nonfinite_steps <= max(1, (W + K) // 100), \
        f'non-finite losses in the timed region: {nonfinite_steps} of {W + K} steps'
    value = BATCH * K * world / (ms * 1e-3)
    if args.dump_outputs and rank == 0:     # before the legs below train the same engine further
        dump_outputs(eng, losses[-1], args.dump_outputs)

    if args.profile:
        print(f'profile run: {ms / K * 1e3:.1f} us/step', flush=True)
        eng.close()
        return
    prof = None
    if world == 1:
        pi0, pi1 = make_plan(n, 64, rng, cs)      # its own plan: the timed one may be shorter than a profile needs
        eng.upload_plan(pi0, pi1, np.full(64, 0.5), stream)
        us = eng.profile_step(48, stream)
        prof = {'sum_us': float(us.sum()), 'phases': [[nm, round(float(u), 2)] for nm, u in zip(eng.phase_names(), us)],
                'note': 'microseconds per phase inside the persistent kernel (GPU global timer at the phase boundaries, grid '
                        'barrier included), averaged over 48 consecutive steps of one launch'}

    # ---------------- end to end with host-resident data
    Ke = max(20, min(K, 300))
    nh = min(n, 200_000)
    host = [d[:nh].cpu().pin_memory() for d in data]
    hb = [[torch.empty((BATCH, d), dtype=torch.float32).pin_memory() for d in DIMS] for _ in range(2)]   # two host slots
    i0e, i1e = make_plan(nh, Ke + 5, rng, cs if nz.max() < nh else np.stack([np.flatnonzero(mask[:nh])[:2]] * 2, 1))
    ti = [torch.from_numpy(i0e), torch.from_numpy(i1e)]

    def e2e_run(first, count):
        """The reference's loop shape (jamie/jamie.py:549-742) with host-resident data: gather the batch rows on the host,
        hand them to the engine, read the step's losses back. N = 1: the engine's asynchronous host-batch API keeps two
        steps in flight, so the host gather of batch k + 1 overlaps step k (also at N > 1 when the step kernel carries the
        gradient exchange); N > 1 with an NCCL / multimem exchange: backward, all-reduce, update."""
        out, pending = None, 0
        for s in range(first, first + count):
            b = hb[s & 1]
            for i in range(2):
                torch.index_select(host[i], 0, ti[i][s], out=b[i])      # the reference's dataset[i][random_batch[i]]
            if world == 1 or gx.mode == 'kernel':   # (N > 1: the step kernel exchanges the gradients itself, same pipeline)
                eng.hostbatch_submit(b[0].data_ptr(), b[1].data_ptr(), i0e[s], i1e[s], 0.5, stream)
                pending += 1
                if pending == 2:
                    out = eng.hostbatch_wait()
                    pending -= 1
            else:
                eng.step_backward_hostbatch(b[0].data_ptr(), b[1].data_ptr(), i0e[s], i1e[s], 0.5, stream)
                gx.all_reduce()
                eng.step_update(stream)
                out = eng.read_losses(2, stream)[s & 1]
        while pending:
            out = eng.hostbatch_wait()
            pending -= 1
        return out

    e2e_run(0, 5)
    sync_all()
    t0 = time.perf_counter()
    out = e2e_run(5, Ke)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    assert np.isfinite(out[4]), f"non-finite loss at the end of the end-to-end leg: {out}"
    e2e_value = BATCH * Ke * world / dt
    h2d = sum(BATCH * d * 4 for d in DIMS) + 2 * BATCH * 4 + 4
    d2h = 8 * 4
    del host

    pred = predict_leg(eng, torch, peaks, stream) if not args.no_predict else None
    if pred is not None and world > 1:      # rows/s of the whole job: every rank imputes its own shard, no collective
        t = torch.tensor([pred['ms'], pred['rows'] / pred['e2e']['value']], device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        pred['value'] = world * pred['rows'] / (float(t[0]) * 1e-3)
        pred['e2e']['value'] = world * pred['e2e']['rows'] / float(t[1])
    line = None
    if rank == 0:
        step_us = ms * 1e3 / K
        roof = {'bound': 'hbm', 'kernel': 'k_step (the whole optimizer step is one persistent kernel)',
                'achieved': ALG_BYTES_PER_STEP / (step_us * 1e-6) / 1e9, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                'frac': ALG_BYTES_PER_STEP / (step_us * 1e-6) / 1e9 / peaks['hbm_gbs'], 'traffic': ncu_traffic('k_step_per_step'),
                'us_per_step': step_us, 'bytes_per_step': ALG_BYTES_PER_STEP, 'peak_source': peaks['source'],
                'note': 'algorithmic bytes of a step = r/w of fp32 params + Adam m, v (6*4*4312194) + gathered inputs '
                        '(SURVEY.md 8d: the step roofline is 16.1 us); traffic = DRAM bytes per step from the committed ncu capture'}
        groof = None
        if prof is not None:
            gem = [(nm, u) for nm, u in prof['phases'] if nm.startswith('gemm') or nm.startswith('dgrad') or nm.startswith('wgrad')]
            gus = sum(u for _, u in gem)
            groof = {'bound': 'tensor', 'achieved': ALG_FLOPS_PER_STEP / (gus * 1e-6) / 1e12, 'peak': peaks['bf16_tflops_sustained'],
                     'unit': 'TFLOP/s', 'frac': ALG_FLOPS_PER_STEP / (gus * 1e-6) / 1e12 / peaks['bf16_tflops_sustained'],
                     'gemm_phases_us': round(gus, 2), 'flops_per_step': ALG_FLOPS_PER_STEP,
                     'note': 'all 12 GEMM phases of a step together: algorithmic FLOPs (one fp32-class product per MAC; the '
                             'kernel issues three fp16 tensor-core passes per product) over their in-kernel time. Since the '
                             'cluster fusion these phases also contain the BatchNorm / dropout / loss tails and their grid '
                             'barriers (the separate element-wise phases are gone), so this is a lower bound of the GEMM rate'}
        fit = None
        if world == 1 and not args.no_fit:
            eng.close()
            del data
            torch.cuda.empty_cache()
            fit = fit_transform_leg(torch)
        cb = None
        if world == 1 and not args.no_cpu_baseline:   # last: importing the reference replaces the `jamie` package in sys.modules
            cb = cpu_baseline()
        line = {
            'metric': 'train cells/sec (fwd+bwd+Adam)', 'value': value, 'unit': 'cells/s', 'n_gpus': world,
            'steps': K, 'warmup': W, 'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f16x2 (fp16 hi/lo split operands, fp32 accumulate: fp32-class products)', 'data': 'synthetic',
            'config': dict(workload_config(world), **({'exchange': ('in-kernel reduce-scatter + all-gather over NVLink peer memory' + (' (NVLS multimem)' if getattr(gx, 'multicast', False) else '') + ', between WGRAD and ADAM of the persistent step kernel' if gx.mode == 'kernel' else gx.mode + ' all-reduce of the flat gradient buffer') + ' (jamie_b200/dp.py)'} if gx is not None else {})),
            'e2e': {'value': e2e_value, 'unit': 'cells/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'steps': Ke, 'note': 'per step: host gather of the batch rows into pinned memory, H2D of rows + cell ids, '
                                         'step kernel, D2H of the 8 loss scalars; jb_hostbatch_submit / jb_hostbatch_wait keep '
                                         'two steps in flight (N = 1)'},
            'e2e_fit_transform': fit,
            'gpu_launches': int(launches), 'launches_per_step': launches / K,
            'roofline': roof, 'gemm_roofline': groof, 'step_profile': prof,
            'modal_predict': pred, 'cpu_baseline': cb, 'clocks': clocks.summary(),
            'final_losses': {k: float(v) for k, v in zip(['KL', 'Rec', 'CosSim', 'F', 'total', 'grad_norm'], losses[-1])},
            'nonfinite_steps': nonfinite_steps,
        }
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    try:
        eng.close()
    except Exception:
        pass


if __name__ == '__main__':
    main()
