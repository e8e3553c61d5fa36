"""CPU tests of the host-side mirror: initial weights, sampler draws, prior handling, preprocessing, metrics, and the
epoch bookkeeping helpers -- checked against the reference fixtures and the oracle."""
import numpy as np
import pytest
import torch

from oracle import jamie_oracle as O
from tests.golden_util import CASES, Golden


@pytest.fixture(autouse=True)
def host_projection():
    """These tests pin the host arithmetic. In a session that also ran GPU tests, the engine of a JAMIE model that was
    never closed stays attached as the process's PCA projector and would take preclass onto the GPU (fp32 class)."""
    from jamie_b200 import utilities as Ut
    attached = Ut._GPU_PROJECTOR
    Ut.set_gpu_projector(None)
    yield
    Ut.set_gpu_projector(attached)


@pytest.mark.parametrize('name', ['diag_drop', 'rep_F', 'zeros_unequal'])
def test_initial_weights_equal_reference(name):
    """Same torch seed + same construction order => bit-identical initial parameters as the reference model."""
    from jamie_b200.model import edModelVar
    G = Golden(name)
    torch.manual_seed(666)
    m = edModelVar(G.meta['col'], G.kw['output_dim'], dropout=G.kw.get('dropout'))
    assert [n for n, _ in m.named_parameters()] == G.param_names
    for got, want in zip(m.packed_parameters(), G.init_params()):
        np.testing.assert_array_equal(got, want)
    assert m.dropout_p == G.meta['dropout']
    for k, v in m.packed_buffers().items():
        np.testing.assert_array_equal(v, G.buffers('init')[k])


def test_layout_matches_oracle_spec():
    from jamie_b200.layout import bn_spec, param_spec
    assert param_spec([512, 39], 32) == O.param_spec([512, 39], 32)
    assert bn_spec([7, 9]) == O.bn_spec([7, 9])
    assert sum(int(np.prod(s)) for _, s in param_spec([512, 512], 32)) == 4312194      # SURVEY.md section 8a


@pytest.mark.parametrize('name', CASES)
def test_sampler_reproduces_reference_draws(name):
    from jamie_b200.jamie import PriorSpec, sample_batch
    G = Golden(name)
    rows, dims, B = G.meta['n'], G.meta['col'], G.meta['batch_size']
    prior = PriorSpec(G['P'] if G.has('P') else None, rows)
    assert prior.sampling_method == G.meta['sampling_method']
    np.random.seed(42)
    for s in range(G.n_steps):
        idx = sample_batch(prior.sampling_method, rows, dims, B, prior.corr_samples)
        data = [G[f'pre{i}'].astype(np.float32) for i in range(2)]
        for i in range(2):
            np.testing.assert_array_equal(data[i][idx[i]], G[f's{s}/x{i}'])


def test_prior_forms_are_equivalent():
    from jamie_b200.jamie import PriorSpec
    import scipy.sparse as sp
    m = (np.arange(10) % 3 == 0).astype(np.float64)
    a = PriorSpec(np.diag(m), [10, 10])
    b = PriorSpec(m, [10, 10])
    c = PriorSpec(sp.diags(m).tocsr(), [10, 10])
    for p in (a, b, c):
        assert p.sampling_method == 'hybrid' and p.dense is None
        np.testing.assert_array_equal(p.diag, m)
        np.testing.assert_array_equal(p.corr_samples, [[0, 0], [3, 3]])
    assert PriorSpec(None, [5, 5]).sampling_method == 'diag'
    assert PriorSpec(None, [5, 4]).sampling_method == 'zeros'
    assert PriorSpec(np.zeros((5, 4)), [5, 4]).sampling_method == 'zeros'
    d = np.zeros((5, 4)); d[1, 2] = 1; d[3, 0] = 2
    pd = PriorSpec(d, [5, 4])
    assert pd.sampling_method == 'hybrid' and pd.dense is not None
    np.testing.assert_array_equal(pd.corr_samples, [[1, 2], [3, 0]])
    np.testing.assert_array_equal(PriorSpec(m, [10, 10]).to_dense(), np.diag(m))


@pytest.mark.parametrize('name', ['diag_drop', 'pca'])
def test_preclass_matches_reference(name):
    from jamie_b200.utilities import LinearPCA, preclass
    G = Golden(name)
    for i in range(2):
        raw = G[f'data{i}']
        if G.kw.get('pca_dim') is not None:
            pca = LinearPCA(G.kw['pca_dim'][i])
            sample = pca.fit_transform(raw)
            # same subspace and sign convention as the reference's sklearn PCA on this (full-SVD) problem
            np.testing.assert_allclose(np.abs(pca.components_ @ G[f'pca_components{i}'].T), np.eye(len(pca.components_)),
                                       atol=1e-6)
            pre = preclass(sample, pca=pca)
            np.testing.assert_allclose(np.abs(pre.transform(raw)), np.abs(G[f'pre{i}']), rtol=1e-6, atol=1e-8)
            np.testing.assert_allclose(pre.inverse_transform(pre.transform(raw)),
                                       pca.inverse_transform(pca.transform(raw)), rtol=1e-9, atol=1e-9)
        else:
            pre = preclass(raw, axis=0)
            np.testing.assert_allclose(pre.transform(raw), G[f'pre{i}'], rtol=1e-12, atol=1e-12)
            np.testing.assert_allclose(pre.inverse_transform(pre.transform(raw)), raw, rtol=1e-9, atol=1e-9)
    const = np.ones((6, 3))
    assert np.all(preclass(const, axis=0).transform(const) == 0)        # NaN -> 0 rule (jamie/utilities.py:669)


def test_constructor_surface_and_validation():
    from jamie import JAMIE
    jm = JAMIE(min_epochs=500)
    assert (jm.batch_size, jm.epoch_DNN, jm.log_DNN, jm.output_dim, jm.manual_seed) == (512, 10000, 500, 32, 666)
    assert jm.pca_dim == [512, 512] and jm.use_f_tilde and jm.min_epochs == 500 and jm.project_mode == 'jamie'
    with pytest.raises(TypeError):
        JAMIE(not_an_argument=1)
    with pytest.raises(Exception, match='distance_mode error'):
        JAMIE(distance_mode='nope').fit_transform(dataset=[np.zeros((4, 3)), np.zeros((4, 3))])
    with pytest.raises(AssertionError, match='Model must be trained'):
        JAMIE().modal_predict(np.zeros((2, 2)), 0)
    # the engine implements edModelVar only: any other model_class is rejected before anything is trained
    with pytest.raises(NotImplementedError, match='model_class'):
        JAMIE(model_class=dict, use_f_tilde=False, pca_dim=None).fit_transform(dataset=[np.random.rand(8, 3), np.random.rand(8, 3)])


def test_metrics():
    """The metrics oracle (oracle/metrics_oracle.py, the checker of the GPU metrics) against the reference's own formulas
    (jamie/evaluation.py:65-85, 114-132; jamie/jamie.py:943-961) restated with the sklearn calls the reference makes."""
    import contextlib
    import io
    from sklearn.metrics import pairwise_distances
    from sklearn.neighbors import KNeighborsClassifier
    from oracle import metrics_oracle as E
    rng = np.random.default_rng(0)
    a = rng.normal(size=(60, 4))
    b = a + 0.4 * rng.normal(size=a.shape)

    def ref_foscttm(x):
        d = pairwise_distances(np.concatenate(x, axis=0), metric='euclidean')
        size = x[0].shape[0]
        cnt = 0
        for i in range(size):
            loc = d[i][size:]
            cnt += np.sum(loc < loc[i])
            loc = d[size + i][:size]
            cnt += np.sum(loc < loc[i])
        return cnt / (2 * size ** 2)

    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        got = E.test_closer([a, b])
    assert buf.getvalue().startswith('foscttm: ')              # the reference prints this line
    assert got == pytest.approx(ref_foscttm([a, b]), abs=1e-12)
    assert E.test_closer([a, a], verbose=False) == 0.0
    assert E.test_closer([a, b], distance_metric=lambda x: pairwise_distances(x, metric='euclidean'), verbose=False) == got
    # label transfer: unequal set sizes and label sets, default k = int(.2 * min(len) / n_classes(concat))
    y0 = rng.integers(0, 3, size=60)
    emb1 = rng.normal(size=(45, 4))
    y1 = rng.integers(1, 4, size=45)
    emb0 = a + np.eye(4)[y0 % 4] * 2
    for k in (None, 1, 5):
        kk = int(.2 * 45 / 4) if k is None else k
        knn = KNeighborsClassifier(n_neighbors=kk).fit(emb1, y1)
        want = float(np.mean(knn.predict(emb0) == y0))
        acc, k_used = E.label_transfer_accuracy([emb0, emb1], [y0, y1], k=k, return_k=True)
        assert k_used == kk and acc == pytest.approx(want, abs=1e-12)
    assert E.test_LabelTA([emb0, emb1], [y0, y1], verbose=False) == E.label_transfer_accuracy([emb0, emb1], [y0, y1], k=5)
    r = E.imputation_correlation(a * 2 + 1, a)
    np.testing.assert_allclose(r, 1.0)
    assert E.mean_feature_r(np.c_[a, a[:, :1]], np.c_[a, np.ones((60, 1))]) == pytest.approx(1.0)


def test_geodesic_distances_properties():
    """unioncom's geodesic_distances as restated in jamie_b200/correspondence.py (third-party, parity unpinned): a
    connected kNN graph gives a symmetric metric with zero diagonal that dominates the euclidean distance; unreachable
    pairs are set to twice the largest finite distance."""
    from sklearn.metrics import pairwise_distances
    from jamie_b200.correspondence import distance_function, geodesic_distances
    rng = np.random.default_rng(3)
    t = np.sort(rng.random(80))
    X = np.stack([np.cos(3 * t), np.sin(3 * t)], 1) + 0.01 * rng.normal(size=(80, 2))
    d = geodesic_distances(X, 40)
    assert d.shape == (80, 80) and np.allclose(d, d.T) and np.all(np.diag(d) == 0) and np.all(np.isfinite(d))
    assert np.all(d >= pairwise_distances(X) - 1e-9)                 # paths are at least as long as the chord
    assert d[0, -1] > 1.3 * np.linalg.norm(X[0] - X[-1])             # along the arc, not across it
    far = np.concatenate([X[:6], X[:6] + 1000.0])                    # two clusters no kNN graph up to kmax connects
    d2 = geodesic_distances(far, 2)
    finite = d2[:6, :6].max()
    assert np.allclose(d2[:6, 6:], 2 * max(finite, d2[6:, 6:].max()))
    np.testing.assert_allclose(distance_function('cosine', 40)(X), pairwise_distances(X, metric='cosine'))
    sp = distance_function('spearman', 40)(rng.normal(size=(5, 30)))
    assert sp.shape == (5, 5) and np.allclose(np.diag(sp), 0)


def test_kl_anneal_and_chunk_bound():
    # anneal midpoint and shape (jamie/jamie.py:630-631)
    assert abs(O.kl_anneal(250, 500, 10000) - 0.5) < 1e-12
    assert O.kl_anneal(0, 0, 100) < 0.01 < O.kl_anneal(100, 0, 100)


def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): exactly one JSON line on stdout with the
    contract's keys; it times the oracle port only (no GPU, no CUDA library)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '2', '--warmup', '3'],
                         capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'cells/s' and d['higher_is_better'] is True and d['value'] > 0
    assert (d['steps'], d['warmup']) == (2, 3) and (d['cpu_baseline']['steps'], d['cpu_baseline']['warmup']) == (2, 3)
    assert d['cpu_baseline']['kind'] in ('reference', 'port') and d['cpu_baseline']['cores'] >= 1
    assert d['e2e'] == {'value': d['value'], 'unit': 'cells/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert d['config']['workload'].startswith('BASELINE configs[3]')


def test_fast_sampler_distribution_and_reference_default():
    """sampler='fast' / 'auto' above 16k cells: an O(batch) draw with the reference's distribution (distinct indices in
    range, hybrid head from the matched pairs); the default path below that size stays the reference's numpy stream."""
    from jamie_b200.jamie import sample_batch
    rows, cols, B = [100_000, 90_000], [512, 512], 512
    rng = np.random.default_rng(7)
    cs = [np.array([11, 22]), np.array([33, 44])]
    np.random.seed(3)
    for method in ('diag', 'zeros', 'hybrid'):
        rb = sample_batch(method, rows, cols, B, cs, fast_rng=rng)
        assert len(rb) == 2 and all(len(r) == B for r in rb)
        for i in range(2):
            tail = rb[i] if method != 'hybrid' else rb[i][np.isin(rb[i], cs[i], invert=True)]
            assert tail.min() >= 0 and tail.max() < rows[0 if method == 'diag' else i]
            assert len(np.unique(tail)) == len(tail)
        if method == 'diag':
            assert rb[0] is rb[1]
        if method == 'hybrid':
            k = B - len(rb[0][np.isin(rb[0], cs[0], invert=True)])
            assert k <= 2 and set(rb[0][:k]) <= set(cs[0]) and set(rb[1][:k]) <= set(cs[1])
    # uniformity: mean of many draws is close to (n - 1) / 2
    draws = np.concatenate([sample_batch('zeros', rows, cols, B, fast_rng=rng)[0] for _ in range(200)])
    assert abs(draws.mean() / (rows[0] - 1) - 0.5) < 0.01
    # replacement sampling (narrow modality) and the default path keep the legacy global generator
    np.random.seed(5)
    a = sample_batch('diag', [300, 300], [39, 512], B, fast_rng=rng)[0]
    np.random.seed(5)
    b = np.random.choice(300, B, replace=True)
    np.testing.assert_array_equal(a, b)
    np.random.seed(6)
    c = sample_batch('zeros', [400, 300], cols, 128)
    np.random.seed(6)
    np.testing.assert_array_equal(c[0], np.random.choice(range(400), 128, replace=False))


def test_chunked_early_stopping_matches_the_epoch_by_epoch_rule():
    """The fit loop enqueues chunks of epochs and samples the next chunk while the GPU runs (its size bounded by the
    largest streak the running chunk can end with): whatever the loss sequence, early stopping fires at the same epoch as
    the reference's epoch-by-epoch rule (jamie/jamie.py:777-792) and always on the last epoch of a chunk."""
    from jamie_b200.jamie import chunk_epochs
    rng = np.random.default_rng(0)
    for trial in range(200):
        epoch_DNN = int(rng.integers(1, 400))
        min_epochs = int(rng.integers(0, 200))
        msi = int(rng.integers(1, 40))
        ldl = int(rng.integers(1, 300))
        use_es = bool(rng.integers(0, 4))
        losses = np.minimum.accumulate(rng.random(epoch_DNN) + 1.0) if trial % 3 else rng.random(epoch_DNN)
        losses = losses + (rng.random(epoch_DNN) < 0.5) * 0.05        # plateaus and regressions

        def rule(epoch, best, streak):          # one epoch of the reference's early-stop bookkeeping
            stop = False
            if epoch > min_epochs:
                if best - losses[epoch] > 1e-8:
                    best, streak = losses[epoch], 0
                else:
                    streak += 1
                stop = streak >= msi and use_es
            return best, streak, stop
        # reference: epoch by epoch
        best, streak, want = np.inf, 0, epoch_DNN
        for ep in range(epoch_DNN):
            best, streak, stop = rule(ep, best, streak)
            if stop:
                want = ep + 1
                break
        # chunked + pipelined, as in JAMIE.project_jamie
        best, streak, epoch, stop = np.inf, 0, 0, False
        n = chunk_epochs(0, 0, min_epochs, msi, use_es, epoch_DNN, ldl)
        while n is not None and not stop:
            assert 1 <= n <= epoch_DNN - epoch and n * ldl <= max(4096, ldl)
            nxt = chunk_epochs(epoch + n, streak + n, min_epochs, msi, use_es, epoch_DNN, ldl) if epoch + n < epoch_DNN else None
            for e_ in range(n):
                best, streak, stop = rule(epoch, best, streak)
                epoch += 1
                if stop:
                    assert e_ == n - 1, 'early stop inside a chunk'
                    break
            n = nxt
        assert epoch == want, (trial, epoch, want)


def test_pca_fit_accepts_sparse_blocks():
    """scipy.sparse inputs (AnnData.X) go through the PCA fit and the projection 16 k densified rows at a time: column sums,
    Gram matrices and projections add up / concatenate over row blocks, so the result equals the dense one (the GPU passes
    are replaced by numpy stand-ins here; the block logic is what is tested)."""
    import scipy.sparse as sp
    from jamie_b200 import pca_fit

    class HostPasses:
        calls = 0

        def pca_colsum(self, X):
            HostPasses.calls += 1
            assert isinstance(X, np.ndarray) and X.dtype == np.float32
            return X.astype(np.float64).sum(0)

        def pca_gram(self, X, mean):
            Xc = X.astype(np.float64) - mean
            return Xc.T @ Xc

        def pca_project(self, X, comp, mean, m, s):
            return ((X.astype(np.float64) - mean) @ comp.T - m) / s

    rng = np.random.default_rng(1)
    X = (rng.random((700, 40)) * (rng.random((700, 40)) < 0.2)).astype(np.float32)       # 80 % zeros
    X[:, :6] += (rng.normal(size=(700, 3)) @ rng.normal(size=(3, 6))).astype(np.float32)
    old = pca_fit.BLOCK_ROWS
    try:
        pca_d, sample_d = pca_fit.fit_transform(HostPasses(), X, 5)
        n_dense = HostPasses.calls
        blocks = list(pca_fit.dense_blocks(sp.csr_matrix(X), 100, 650, rows=256))
        assert [b[0] for b in blocks] == [100, 356, 612] and blocks[-1][1].shape == (38, 40)
        np.testing.assert_array_equal(np.concatenate([b[1] for b in blocks]), X[100:650])
        HostPasses.calls = 0
        pca_fit.dense_blocks.__defaults__ = (0, None, 256)      # small blocks so that several are summed
        pca_s, sample_s = pca_fit.fit_transform(HostPasses(), sp.csr_matrix(X), 5)
        assert HostPasses.calls == 3 and n_dense == 1
    finally:
        pca_fit.dense_blocks.__defaults__ = (0, None, old)
    np.testing.assert_allclose(pca_s.components_, pca_d.components_, atol=1e-10)
    np.testing.assert_allclose(pca_s.explained_variance_, pca_d.explained_variance_, rtol=1e-10)
    np.testing.assert_allclose(sample_s, sample_d, atol=1e-9)
