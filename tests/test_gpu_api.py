"""End-to-end through the reference-facing Python API (jamie.JAMIE) on the GPU."""
import os

import numpy as np
import pytest

from tests import parity_util as U
from tests.golden_util import GOLDEN_DIR

pytestmark = pytest.mark.gpu


def _mmdma_like(n=300, dims=(200, 100), seed=0):
    rng = np.random.default_rng(seed)
    t = rng.random(n) * 2 - 1
    branch = rng.integers(0, 3, n)
    lat = np.stack([t, t ** 2 * (branch == 0) + t * (branch == 1) - t * (branch == 2), np.sin(3 * t)], 1)
    data = []
    for d in dims:
        W = rng.normal(size=(3, d))
        data.append(lat @ W + 0.05 * rng.normal(size=(n, d)))
    return data, branch


def test_fit_transform_end_to_end(capsys):
    from jamie import JAMIE
    data, labels = _mmdma_like()
    np.random.seed(42)
    jm = JAMIE(output_dim=16, batch_size=128, pca_dim=[32, 32], epoch_DNN=400, min_epochs=100, log_DNN=100,
               use_f_tilde=False, debug=True, log_debug=200)
    emb = jm.fit_transform(dataset=data)
    out = capsys.readouterr().out
    assert 'use random seed: 666' in out and 'Train coupled autoencoders' in out and 'Finished Mapping!' in out
    assert 'epoch:[400/400]: loss:' in out and 'JAMIE Done!' in out
    assert emb[0].shape == (300, 16) and emb[1].shape == (300, 16)
    assert set(jm.loss_history) == {'KL', 'Rec', 'CosSim', 'F'} and len(jm.loss_history['Rec']) == jm.epochs_run
    assert jm.sampling_method == 'diag'
    assert np.mean(jm.loss_history['Rec'][-20:]) < 0.5 * np.mean(jm.loss_history['Rec'][:5])
    fos = jm.test_closer(emb)
    lta = jm.test_LabelTA(emb, [labels, labels], k=5)
    assert fos < 0.1 and lta > 0.8, (fos, lta)
    # fit_transform's return equals transform_one / transform on the training data (SURVEY App. A.7)
    for i in range(2):
        np.testing.assert_array_equal(jm.transform_one(data[i], i), emb[i])
    np.testing.assert_array_equal(jm.transform(data)[1], emb[1])
    # imputation: held-in correlation per feature is high on this noiseless-ish manifold
    from jamie_b200.evaluation import imputation_correlation
    pred1 = jm.modal_predict(data[0], 0)
    assert pred1.shape == data[1].shape and pred1.dtype == np.float64
    assert np.nanmean(imputation_correlation(pred1, data[1])) > 0.7
    jm.engine.close()


def test_ingest_pca_projection_runs_on_the_engine():
    """SURVEY 8(a17): ``preclass.transform`` / ``inverse_transform`` (jamie/utilities.py:660-678) reach jb_pca_project /
    jb_pca_inverse from the product path (ingest in fit_transform, modal_predict in both directions) and agree with the
    reference's float64 host arithmetic to fp32 rounding."""
    from jamie import JAMIE
    from jamie_b200 import utilities as Ut
    data, _ = _mmdma_like(n=200, dims=(150, 90), seed=3)
    jm = JAMIE(output_dim=8, batch_size=64, pca_dim=[24, 20], epoch_DNN=20, min_epochs=5, use_f_tilde=False)
    jm.fit_transform(dataset=data)
    eng = jm.engine
    assert Ut._GPU_PROJECTOR is eng
    l0 = eng.launch_count()
    gpu_pre = [jm.model.preprocessing[i](data[i]) for i in range(2)]
    assert eng.launch_count() > l0                                   # kernels of this engine did the projection
    imp_gpu = jm.modal_predict(data[0], 0)
    Ut.set_gpu_projector(None)                                       # the reference's host path (sklearn, float64)
    try:
        host_pre = [jm.model.preprocessing[i](data[i]) for i in range(2)]
        for i in range(2):
            assert gpu_pre[i].shape == host_pre[i].shape and gpu_pre[i].dtype == np.float64
            assert np.abs(gpu_pre[i] - host_pre[i]).max() < 2e-5 * max(1.0, np.abs(host_pre[i]).max())
            np.testing.assert_allclose(jm.dataset[i], host_pre[i], atol=2e-5 * max(1.0, np.abs(host_pre[i]).max()))
        imp_host = jm.modal_predict(data[0], 0)                      # host pre-processing and inverse, same GPU network
    finally:
        Ut.set_gpu_projector(eng)
    assert U.rel(imp_gpu, imp_host) < 1e-4
    jm.engine.close()
    assert Ut._GPU_PROJECTOR is None


def test_save_load_roundtrip(tmp_path):
    from jamie import JAMIE
    data, _ = _mmdma_like(n=120, dims=(60, 40), seed=1)
    jm = JAMIE(output_dim=8, batch_size=64, pca_dim=[16, 16], epoch_DNN=30, min_epochs=10, use_f_tilde=False)
    jm.fit_transform(dataset=data)
    f = str(tmp_path / 'model.h5')
    jm.save_model(f)
    assert open(f, 'rb').read(4) == b'PK\x03\x04'           # torch zip archive, like the reference's files
    jm2 = JAMIE()
    jm2.load_model(f)
    for i in range(2):
        np.testing.assert_array_equal(jm2.modal_predict(data[i], i), jm.modal_predict(data[i], i))
        np.testing.assert_array_equal(jm2.transform_one(data[i], i), jm.transform_one(data[i], i))
    # the module tree is the reference's
    keys = list(jm2.model.state_dict().keys())
    assert keys[0] == 'sigma' and 'encoders.0.0.weight' in keys and 'decoders.1.8.bias' in keys
    assert 'encoders.0.1.running_mean' in keys and len(keys) == 45 + 24
    jm.engine.close()
    jm2.engine.close()


def test_load_reference_checkpoint():
    """A file written by the reference's own save_model loads here and predicts what the reference predicted."""
    from jamie import JAMIE
    io = np.load(os.path.join(GOLDEN_DIR, 'ref_checkpoint_io.npz'))
    jm = JAMIE()
    jm.load_model(os.path.join(GOLDEN_DIR, 'ref_checkpoint.h5'))
    for i in range(2):
        got = jm.modal_predict(io[f'data{i}'], i)
        assert U.rel(got, io[f'pred{i}']) < 3e-3
        assert U.rel(jm.transform_one(io[f'data{i}'], i), io[f'tone{i}']) < 3e-3
    jm.engine.close()


def test_early_stop_fires_at_the_epoch_the_reference_rule_gives():
    """A run that really stops early (the chunks of epochs the fit loop enqueues never cross the stop decision): with one
    batch per epoch `best_batch_loss` is the epoch's total loss = the sum of the four `loss_history` entries, so the
    reference's bookkeeping (jamie/jamie.py:777-792) can be replayed on the recorded history and must stop where the run did."""
    from jamie import JAMIE
    data, _ = _mmdma_like(n=100, dims=(60, 40), seed=3)
    np.random.seed(7)
    kw = dict(min_epochs=30, min_increment=2e-2, max_steps_without_increment=6, epoch_DNN=3000)
    jm = JAMIE(output_dim=8, batch_size=128, pca_dim=None, use_f_tilde=False, log_DNN=10 ** 6, **kw)
    jm.fit_transform(dataset=data)
    ran = len(jm.loss_history['KL'])
    jm.engine.close()
    assert jm.epochs_run == ran
    total = np.sum([np.asarray(jm.loss_history[k], np.float64) for k in ('KL', 'Rec', 'CosSim', 'F')], axis=0)
    best, streak, want = np.inf, 0, kw['epoch_DNN']
    for epoch in range(len(total)):
        if epoch > kw['min_epochs']:
            if best - total[epoch] > kw['min_increment']:
                best, streak = total[epoch], 0
            else:
                streak += 1
            if streak >= kw['max_steps_without_increment']:
                want = epoch + 1
                break
    assert kw['min_epochs'] + kw['max_steps_without_increment'] < ran < kw['epoch_DNN'], ran     # it did stop early
    assert ran == want, (ran, want)
