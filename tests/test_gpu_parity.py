"""GPU parity tests: the CUDA engine, called through the C ABI, against (a) fixtures recorded from the real reference
and (b) the numpy oracle on seeded inputs at the headline sizes.  north_star asks for 1e-3 relative on per-step losses
and gradients with injected eps / dropout masks / batch indices.  Round 2: every GEMM of the step (forward, dgrad AND
wgrad) runs the three-pass fp16-split product (hgemm.cuh, fp32-class), everything else is fp32, so the engine agrees
with the fp32 oracle to ~1e-6 (profiles/parity_r2.md lists the measured per-tensor errors of every shape) and the
tolerances below are 5x .. 10x TIGHTER than north_star's.  Against the recorded reference fixtures the bound is the
reference's own fp32 noise (oracle vs reference: up to 2e-4 per tensor, tests/test_oracle_golden.py): 1e-3."""
import numpy as np
import pytest

from oracle import jamie_oracle as O
from tests import parity_util as U
from tests.golden_util import CASES, Golden

pytestmark = pytest.mark.gpu

LOSS_RTOL = 1e-4
GRAD_RTOL = 2e-4      # per-tensor ||g - g_ref|| / ||g_ref|| vs the oracle (measured <= 3e-6, profiles/parity_r2.md)
FWD_RTOL = 1e-4       # forward taps vs the oracle (measured <= 6e-7)
REF_RTOL = 1e-3       # vs values recorded from the reference itself (north_star's tolerance)


def _engine(dims, L, B, p, **kw):
    from jamie_b200.engine import Engine
    return Engine(dims, L, B, p, **kw)


def _check_grads(spec, got, want, corr_nonzero, rtol=GRAD_RTOL):
    noise = set(U.PRE_BN_BIAS)
    if not corr_nonzero:
        noise.add('sigma')
    worst = 0.0
    for (n, _), g, w in zip(spec, got, want):
        if n in noise:
            assert np.abs(g).max() < 1e-5, n
            continue
        r = U.rel(g, w)
        worst = max(worst, r)
        assert r < rtol, (n, r)
    return worst


@pytest.mark.parametrize('name', CASES)
def test_reference_fixture_replay(name):
    """Every recorded reference step: same inputs, same randomness -> same losses, gradients, updated parameters."""
    G = Golden(name)
    kw = G.kw
    dims, L, B, rows = G.meta['col'], kw['output_dim'], G.meta['batch_size'], G.meta['n']
    lw = kw.get('loss_weights')
    pf = kw.get('PF_Ratio') or 1
    eng = _engine(dims, L, B, G.meta['dropout'], loss_weights=lw, pf_ratio=pf)
    eng.set_dist_method(kw.get('dist_method', 'euclidean'))
    eng.set_params(G.init_params())
    eng.set_bn_stats(G.buffers('init'))
    data = [G[f'pre{i}'].astype(np.float32) for i in range(2)]
    for i in range(2):
        eng.set_dataset(i, data[i])
    P = G.P_dense()
    method = O.sampling_method(P)
    if G.has('P') or rows[0] == rows[1]:
        if np.count_nonzero(P) == np.count_nonzero(np.diagonal(P)) and P.shape[0] == P.shape[1]:
            eng.set_prior_diag(np.diagonal(P))
        else:
            eng.set_prior_dense(P)
    else:
        eng.set_prior_diag(None)
    eng.set_f_dense(G['F'] if G.has('F') else None)
    corr_samples = np.argwhere(P > 0) if method == 'hybrid' else None
    len_dl = max(int(max(rows) / kw['batch_size']), 1)
    np.random.seed(42)
    idx = [O.sample_batch(method, rows, dims, B, corr_samples) for _ in range(G.n_steps)]
    anneal = [O.kl_anneal(s // len_dl, kw['min_epochs'], kw['epoch_DNN']) for s in range(G.n_steps)]
    eng.upload_plan(np.stack([i[0] for i in idx]), np.stack([i[1] for i in idx]), np.array(anneal))
    names = ['KL', 'Rec', 'CosSim', 'F']
    for s in range(G.n_steps):
        eng.inject(G.eps(s), G.masks(s))
        # start each step from the reference's exact state so that steps are pinned independently
        if s > 0:
            eng.set_params(G.params_after(s - 1))
        eng.train_steps(1)
        ls = eng.read_losses(s + 1)[s]
        np.testing.assert_allclose(eng.debug_read('corr', (B, B)), G[f's{s}/corr'], rtol=1e-6, atol=1e-7)
        for i in range(2):
            assert U.rel(eng.debug_read(f'z{i}', (B, L)), G[f's{s}/z{i}']) < REF_RTOL
            assert U.rel(eng.debug_read(f'c{i}', (B, L)), G[f's{s}/c{i}']) < REF_RTOL
            assert U.rel(eng.debug_read(f'xhat{i}', (B, dims[i])), G[f's{s}/xhat{i}']) < REF_RTOL
        if (s + 1) % len_dl == 0:
            for k, nm in enumerate(names):
                want = G[f'loss_history/{nm}'][s // len_dl] / (lw[k] if lw else 1)
                # CosSim: the reference's cdist route leaves fp32 cancellation noise ~1e-7 (|z|^2 + |c|^2) per row
                # (SURVEY.md App. B-16): absolute floor 1e-4 on that term only
                assert abs(ls[k] - want) <= REF_RTOL * abs(want) + (1e-4 if nm == 'CosSim' else 1e-7), (nm, ls[k], want)
        _check_grads(eng.spec, eng.get_grads(), G.grads(s), np.abs(G[f's{s}/corr']).sum() > 0, rtol=REF_RTOL)
        assert abs(ls[5] - float(G[f's{s}/total_norm'])) < REF_RTOL * ls[5]
    bn = eng.get_bn_stats()
    for k, v in G.buffers(f's{G.n_steps - 1}').items():
        if k.endswith('num_batches_tracked'):
            assert int(bn[k]) == int(v)
        else:
            np.testing.assert_allclose(bn[k], v, rtol=REF_RTOL, atol=1e-4)
    eng.close()


SHAPES = [
    # dims, L, B, p, prior, F
    ([512, 512], 32, 512, 0.6, 'half', False),      # headline (BASELINE configs 2 and 4)
    ([512, 39], 32, 512, 0.6, 'eye_rep', False),    # Patch-seq-like (config 3): duplicates from replacement sampling
    ([2000, 1000], 32, 300, 0.6, 'eye', False),     # MMD-MA without PCA (config 1)
    ([96, 64], 8, 64, 0.0, 'zeros', True),          # no dropout, zero prior, dense F with PF_Ratio < 1
    ([130, 70], 17, 50, 0.3, 'dense', True),        # odd everything: widths, latent, batch
    ([96, 64], 8, 640, 0.3, 'eye', False),          # B > 512: the unfused BatchNorm / reconstruction / reparam phases
]


@pytest.mark.parametrize('dims,L,B,p,prior,use_f', [SHAPES[0], SHAPES[4]])
def test_step_vs_oracle_cosine(dims, L, B, p, prior, use_f):
    """dist_method='cosine' (jamie/jamie.py:485-494): the headline shape on the merged-latent path (no F) and the odd
    shape on the LATLOSS / LATBC path (dense F)."""
    test_step_vs_oracle(dims, L, B, p, prior, use_f, dist_method='cosine')


@pytest.mark.parametrize('dims,L,B,p,prior,use_f', SHAPES)
def test_step_vs_oracle(dims, L, B, p, prior, use_f, dist_method='euclidean'):
    n = 2 * B if prior != 'eye_rep' else B
    rng = np.random.default_rng(5)
    data = U.synth_pair(n, dims, seed=1)
    params = U.torch_like_init(dims, L, seed=2)
    lw = [1, 2, 0.5, 3] if use_f else None
    pf = 0.7 if use_f else 1.0
    eng = _engine(dims, L, B, p, loss_weights=lw, pf_ratio=pf)
    eng.set_dist_method(dist_method)
    eng.set_params(params)
    for i in range(2):
        eng.set_dataset(i, data[i])
    if prior in ('half', 'eye', 'eye_rep', 'zeros'):
        m = {'half': (rng.random(n) < 0.5), 'eye': np.ones(n), 'eye_rep': np.ones(n), 'zeros': np.zeros(n)}[prior]
        m = m.astype(np.float32)
        eng.set_prior_diag(m if m.any() else None)
        P = np.diag(m)
    else:
        P = (rng.random((n, n)) * (rng.random((n, n)) < 0.1)).astype(np.float32)
        eng.set_prior_dense(P)
    Fm = (rng.random((n, n)) * (rng.random((n, n)) < 0.05)).astype(np.float32) if use_f else None
    eng.set_f_dense(Fm)
    Fd = np.zeros((n, n), np.float32) if Fm is None else Fm
    orc = O.OracleModel(dims, L, dropout=p, params=params, dist_method=dist_method)
    rep = prior == 'eye_rep'
    i0 = rng.choice(n, B, replace=rep)
    i1 = i0.copy() if prior in ('eye', 'eye_rep') else np.concatenate([i0[:B // 2], rng.choice(n, B - B // 2, replace=False)])
    eng.upload_plan(i0[None], i1[None], np.array([0.37]))
    eps, masks = U.draw_randomness(B, dims, L, p, seed=11)
    eng.inject(eps, masks)
    eng.train_steps(1)
    ls = eng.read_losses(1)[0]
    x = [data[0][i0], data[1][i1]]
    Pb, Fb = O.corr_block(P, i0, i1), O.corr_block(Fd, i0, i1)
    corr = (np.float32(pf) * Pb + np.float32(1 - pf) * Fb).astype(np.float32)
    ols, ograds, otot, fw = orc.train_step(x, corr, Fb, eps, masks, 0.37, lw)
    np.testing.assert_allclose(eng.debug_read('corr', (B, B)), corr, rtol=1e-6, atol=1e-7)
    taps = U.oracle_taps(fw, orc)
    for key, want in taps.items():
        assert U.rel(eng.debug_read(key, want.shape), want) < FWD_RTOL, key
    for k in range(4):
        assert abs(ls[k] - float(ols[k])) <= LOSS_RTOL * abs(float(ols[k])) + 1e-6, (k, ls[k], ols[k])
    assert abs(ls[5] - otot) < LOSS_RTOL * otot
    worst = _check_grads(eng.spec, eng.get_grads(), [ograds[nm] for nm, _ in orc.spec], np.abs(corr).sum() > 0)
    print(f'dims {dims} worst per-tensor grad rel err {worst:.2e}')
    # post-Adam parameters (first step: update = lr * sign(g) up to eps; compare with an absolute tolerance)
    noise = U.PRE_BN_BIAS | ({'sigma'} if not np.abs(corr).sum() else set())
    for (nm, _), got, want in zip(orc.spec, eng.get_params(), orc.param_list()):
        if nm in noise:
            continue
        bad = np.abs(got - want) > 2e-4
        assert bad.mean() < 2e-3, (nm, bad.mean())     # sign flips of near-zero gradients only
    eng.close()


def test_large_logvar_dynamic_operand_scale():
    """fp16 operand planes overflow at 65504; the latent c and d[mu | logvar] are unbounded (z = mu + exp(logvar / 2) eps:
    the 1M-cell benchmark reached |z| = 1e5 within 60 steps). The step kernel rescales those two operands by an exact,
    dynamically chosen power of two (stepk.cuh: sk_dyn_scale); here a logvar bias of 24 drives |z| past 1e5 and the
    step must still agree with the fp32 oracle."""
    dims, L, B, p = [96, 64], 8, 64, 0.3
    n = 2 * B
    rng = np.random.default_rng(15)
    data = U.synth_pair(n, dims, seed=31)
    params = U.torch_like_init(dims, L, seed=32)
    spec = O.param_spec(dims, L)
    names = [nm for nm, _ in spec]
    params[names.index('fc_vars.1.bias')][:] = 24.0
    eng = _engine(dims, L, B, p)
    eng.set_params(params)
    for i in range(2):
        eng.set_dataset(i, data[i])
    m = (rng.random(n) < 0.5).astype(np.float32)
    eng.set_prior_diag(m)
    eng.set_f_dense(None)
    orc = O.OracleModel(dims, L, dropout=p, params=params)
    i0 = rng.choice(n, B, replace=False)
    i1 = np.concatenate([i0[:B // 2], rng.choice(n, B - B // 2, replace=False)])
    eng.upload_plan(i0[None], i1[None], np.array([0.5]))
    eps, masks = U.draw_randomness(B, dims, L, p, seed=33)
    eng.inject(eps, masks)
    eng.train_steps(1)
    ls = eng.read_losses(1)[0]
    x = [data[0][i0], data[1][i1]]
    P = np.diag(m)
    Pb = O.corr_block(P, i0, i1)
    Fb = np.zeros_like(Pb)
    ols, ograds, otot, fw = orc.train_step(x, Pb.astype(np.float32), Fb, eps, masks, 0.5, None)
    assert np.abs(fw['c'][1]).max() > 65504.0          # the case really leaves fp16's range
    taps = U.oracle_taps(fw, orc)
    for key, want in taps.items():
        assert U.rel(eng.debug_read(key, want.shape), want) < 1e-3, key
    assert np.all(np.isfinite(ls[:6]))
    for k in range(4):
        assert abs(ls[k] - float(ols[k])) <= 1e-3 * abs(float(ols[k])) + 1e-6, (k, ls[k], ols[k])
    assert abs(ls[5] - otot) < 1e-3 * otot
    _check_grads(eng.spec, eng.get_grads(), [ograds[nm] for nm, _ in orc.spec], True, rtol=1e-3)
    eng.close()


def _post_adam_check(spec, got, want, corr_nonzero=True):
    noise = U.PRE_BN_BIAS | (set() if corr_nonzero else {'sigma'})
    for (nm, _), g, w in zip(spec, got, want):
        if nm in noise:
            continue
        bad = np.abs(g - w) > 2e-4
        assert bad.mean() < 2e-3, (nm, bad.mean())     # sign flips of near-zero gradients only (first Adam step = lr * sign)


def test_data_parallel_step_equals_averaged_gradient_update():
    """SURVEY 8(e): R ranks == one update with the gradient averaged over the ranks, per-rank BatchNorm statistics.
    Two engines (world_size = 2) play the two ranks on one GPU: each runs jb_step_backward on its own shard / batch /
    randomness, the flat gradient buffers are summed in place (what the NCCL all-reduce does), each runs
    jb_step_update (which scales by 1 / world_size, clips the AVERAGED gradient's norm and applies Adam). Both ranks must
    end with bit-identical parameters, equal to the oracle's clip + Adam on the averaged oracle gradients."""
    import torch
    dims, L, B, p, R = [96, 64], 8, 64, 0.3, 2
    n = R * 2 * B
    rng = np.random.default_rng(40)
    data = U.synth_pair(n, dims, seed=41)
    params = U.torch_like_init(dims, L, seed=42)
    m = (rng.random(n) < 0.5).astype(np.float32)
    orc = O.OracleModel(dims, L, dropout=p, params=params)
    engines, ograds, olosses = [], [], []
    for r in range(R):
        lo, hi = r * n // R, (r + 1) * n // R
        eng = _engine(dims, L, B, p, world_size=R)
        eng.set_params(params)
        for i in range(2):
            eng.set_dataset(i, data[i][lo:hi])
        eng.set_prior_diag(m[lo:hi])
        eng.set_f_dense(None)
        i0 = rng.choice(hi - lo, B, replace=False)
        i1 = np.concatenate([i0[:B // 2], rng.choice(hi - lo, B - B // 2, replace=False)])
        eng.upload_plan(i0[None], i1[None], np.array([0.4]))
        eps, masks = U.draw_randomness(B, dims, L, p, seed=50 + r)
        eng.inject(eps, masks)
        eng.step_backward()
        engines.append(eng)
        x = [data[0][lo:hi][i0], data[1][lo:hi][i1]]
        Pb = O.corr_block(np.diag(m[lo:hi]), i0, i1).astype(np.float32)
        fw = orc.forward_train(x, Pb, eps, masks, update_buffers=False)
        olosses.append(orc.losses(fw, np.zeros_like(Pb), 0.4))
        ograds.append(orc.backward(fw, np.zeros_like(Pb), 0.4, [1, 1, 1, 1]))
    gts = [e.grad_tensor() for e in engines]
    torch.cuda.synchronize()
    total = gts[0] + gts[1]
    for g in gts:
        g.copy_(total)                                  # all-reduce (SUM) of the flat gradient buffer + loss tail
    torch.cuda.synchronize()
    for e in engines:
        e.step_update()
    avg = {k: ((ograds[0][k].astype(np.float64) + ograds[1][k]) / R).astype(np.float32) for k in ograds[0]}
    onorm = orc.clip_adam(avg)
    got = [e.get_params() for e in engines]
    for a, b in zip(got[0], got[1]):
        np.testing.assert_array_equal(a, b)            # every rank applies the same update
    _check_grads(engines[0].spec, [g / R for g in engines[0].get_grads()], [avg[nm] for nm, _ in orc.spec], True)
    for e in engines:
        ls = e.read_losses(1)[0]
        assert abs(ls[5] - onorm) < LOSS_RTOL * onorm  # clip norm of the averaged gradient
    for r in range(R):
        ls = engines[r].read_losses(1)[0]
        for k in range(4):
            assert abs(ls[k] - float(olosses[r][k])) <= LOSS_RTOL * abs(float(olosses[r][k])) + 1e-6
    _post_adam_check(orc.spec, got[0], orc.param_list())
    for e in engines:
        e.close()


def test_batch_step_false_accumulates_over_the_epoch():
    """``batch_step=False`` (jamie/jamie.py:744-749): gradients of every batch of the epoch accumulate, ONE clip + Adam
    step per epoch, Adam's step count advances once per epoch (not once per backward pass)."""
    dims, L, B, p, nb = [80, 48], 8, 32, 0.25, 3
    n = 4 * B
    rng = np.random.default_rng(60)
    data = U.synth_pair(n, dims, seed=61)
    params = U.torch_like_init(dims, L, seed=62)
    m = np.ones(n, np.float32)
    eng = _engine(dims, L, B, p)
    eng.set_params(params)
    for i in range(2):
        eng.set_dataset(i, data[i])
    eng.set_prior_diag(m)
    eng.set_f_dense(None)
    orc = O.OracleModel(dims, L, dropout=p, params=params)
    idx = np.stack([rng.choice(n, B, replace=False) for _ in range(2 * nb)])
    eng.upload_plan(idx, idx, np.full(2 * nb, 0.3))
    for epoch in range(2):
        acc = None
        for b in range(nb):
            s = epoch * nb + b
            eps, masks = U.draw_randomness(B, dims, L, p, seed=70 + s)
            eng.set_grad_accumulate(b != 0)
            eng.inject(eps, masks)
            eng.step_backward()
            x = [data[0][idx[s]], data[1][idx[s]]]
            Pb = np.eye(B, dtype=np.float32)
            fw = orc.forward_train(x, Pb, eps, masks)
            orc.losses(fw, np.zeros_like(Pb), 0.3)
            g = orc.backward(fw, np.zeros_like(Pb), 0.3, [1, 1, 1, 1])
            acc = g if acc is None else {k: acc[k] + g[k] for k in g}
        _check_grads(eng.spec, eng.get_grads(), [acc[nm] for nm, _ in orc.spec], True)
        eng.step_update()
        onorm = orc.clip_adam(acc)
        assert eng.get_adam_state()[2] == epoch + 1 == orc.adam_t
        assert abs(eng.read_losses(2 * nb)[epoch * nb + nb - 1][5] - onorm) < LOSS_RTOL * onorm
    # second epoch's update is not a sign step any more: compare the parameters directly
    for (nm, _), got, want in zip(orc.spec, eng.get_params(), orc.param_list()):
        if nm in U.PRE_BN_BIAS:
            continue
        assert np.abs(got - want).max() < 3e-4, nm
        assert U.rel(got - np.asarray(params[[k for k, _ in orc.spec].index(nm)]), want - np.asarray(params[[k for k, _ in orc.spec].index(nm)])) < 0.05, nm
    eng.close()


def test_philox_statistics_and_determinism():
    dims, L, B, p = [256, 128], 16, 256, 0.6
    n = 1024
    data = U.synth_pair(n, dims, seed=3)
    params = U.torch_like_init(dims, L, seed=4)
    rng = np.random.default_rng(0)
    idx = np.stack([rng.choice(n, B, replace=False) for _ in range(6)])
    out = []
    for rep_ in range(2):
        eng = _engine(dims, L, B, p, seed=123)
        eng.set_params(params)
        for i in range(2):
            eng.set_dataset(i, data[i])
        eng.set_prior_diag(np.ones(n, np.float32))
        eng.set_f_dense(None)
        eng.upload_plan(idx, idx, np.full(6, 0.5))
        eng.train_steps(6)
        out.append(eng.read_losses(6).copy())
        if rep_ == 0:
            h1 = eng.debug_read('h1_0', (B, 2 * dims[0]))
            eps = eng.debug_read('eps0', (B, L))
            keep = (h1 != 0).mean()
            assert abs(keep - (1 - p)) < 0.01, keep
            assert abs(eps.mean()) < 0.06 and abs(eps.std() - 1) < 0.06
        eng.close()
    np.testing.assert_array_equal(out[0], out[1])       # bit-reproducible: fixed-order reductions, counter-based RNG
    assert np.all(np.isfinite(out[0][:, :6]))


def test_training_reduces_loss():
    dims, L, B, p = [128, 96], 16, 128, 0.2
    n = 512
    data = U.synth_pair(n, dims, seed=7)
    eng = _engine(dims, L, B, p, seed=1)
    eng.set_params(U.torch_like_init(dims, L, seed=8))
    for i in range(2):
        eng.set_dataset(i, data[i])
    eng.set_prior_diag(np.ones(n, np.float32))
    eng.set_f_dense(None)
    rng = np.random.default_rng(0)
    steps = 300
    idx = np.stack([rng.choice(n, B, replace=False) for _ in range(steps)])
    eng.upload_plan(idx, idx, np.full(steps, 0.5))
    eng.train_steps(steps)
    ls = eng.read_losses(steps)
    assert ls[-20:, 1].mean() < 0.6 * ls[:20, 1].mean()     # reconstruction loss
    assert ls[-20:, 4].mean() < ls[:20, 4].mean()
    eng.close()


def test_split_step_equals_fused_step():
    """jb_step_backward + jb_step_update (the data-parallel split) == jb_train_steps at world_size 1."""
    dims, L, B, p = [64, 48], 8, 32, 0.5
    n = 128
    data = U.synth_pair(n, dims, seed=2)
    params = U.torch_like_init(dims, L, seed=3)
    rng = np.random.default_rng(1)
    idx = np.stack([rng.choice(n, B, replace=False) for _ in range(4)])
    res = []
    for split in (False, True):
        eng = _engine(dims, L, B, p, seed=9)
        eng.set_params(params)
        for i in range(2):
            eng.set_dataset(i, data[i])
        eng.set_prior_diag(np.ones(n, np.float32))
        eng.set_f_dense(None)
        eng.upload_plan(idx, idx, np.full(4, 0.2))
        if split:
            for _ in range(4):
                eng.step_backward()
                eng.step_update()
        else:
            eng.train_steps(4)
        res.append((eng.read_losses(4).copy(), eng.get_params(as_list=False)))
        eng.close()
    np.testing.assert_array_equal(res[0][0][:, :5], res[1][0][:, :5])     # the losses are bit-identical
    # The clip norm is summed differently: a launch that holds the whole step takes per-work-item partial sums from the
    # weight-gradient epilogues, the split path (whose gradient buffer may have been all-reduced in between) sweeps the
    # buffer. Same value to ~1e-7 relative, so the clip coefficient and the parameters agree to the last bit or two.
    np.testing.assert_allclose(res[0][0][:, 5], res[1][0][:, 5], rtol=1e-6)
    np.testing.assert_allclose(res[0][1], res[1][1], rtol=0, atol=1e-6)


def test_hostbatch_async_equals_sync_and_resident():
    """Host-resident data: the asynchronous two-slot API (jb_hostbatch_submit / jb_hostbatch_wait), the synchronous
    jb_train_step_hostbatch and the device-resident plan path run the same steps: identical losses and parameters
    (same Philox counters: the step index, not the slot, keys the streams)."""
    import torch
    dims, L, B, p, n, steps = [96, 64], 8, 64, 0.4, 256, 5
    data = U.synth_pair(n, dims, seed=21)
    params = U.torch_like_init(dims, L, seed=22)
    rng = np.random.default_rng(23)
    idx = np.stack([rng.choice(n, B, replace=False) for _ in range(steps)])
    m = (np.arange(n) % 3 != 0).astype(np.float32)
    host = [torch.from_numpy(d).pin_memory() for d in data]
    res = []
    for mode in ('resident', 'sync', 'async'):
        eng = _engine(dims, L, B, p, seed=5)
        eng.set_params(params)
        eng.set_prior_diag(m)
        eng.set_f_dense(None)
        if mode == 'resident':
            for i in range(2):
                eng.set_dataset(i, data[i])
            eng.upload_plan(idx, idx, np.full(steps, 0.3))
            eng.train_steps(steps)
            losses = eng.read_losses(steps)[:, :6].copy()
        else:
            bufs = [[torch.empty((B, d), dtype=torch.float32).pin_memory() for d in dims] for _ in range(2)]
            losses, pending = [], 0
            for s in range(steps):
                b = bufs[s & 1]
                for i in range(2):
                    torch.index_select(host[i], 0, torch.from_numpy(idx[s]), out=b[i])
                if mode == 'sync':
                    losses.append(eng.train_step_hostbatch(b[0].data_ptr(), b[1].data_ptr(), idx[s], idx[s], 0.3)[:6])
                else:
                    eng.hostbatch_submit(b[0].data_ptr(), b[1].data_ptr(), idx[s], idx[s], 0.3)
                    pending += 1
                    if pending == 2:
                        losses.append(eng.hostbatch_wait()[:6])
                        pending -= 1
            while pending:
                losses.append(eng.hostbatch_wait()[:6])
                pending -= 1
            losses = np.stack(losses)
        res.append((losses, np.concatenate([t.ravel() for t in eng.get_params()])))
        eng.close()
    for other in res[1:]:
        np.testing.assert_array_equal(other[0], res[0][0])
        np.testing.assert_array_equal(other[1], res[0][1])
    with pytest.raises(RuntimeError, match='no host-batch step in flight'):
        eng = _engine(dims, L, B, p)
        eng.hostbatch_wait()

