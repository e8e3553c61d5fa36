"""silhouette_samples / silhouette_score on the GPU (jb_silhouette: csrc/silhouette.cuh): the device's intra / inter sums
equal the float64 reference's (tests/silhouette_oracle.py) across tile (64-row) and chunk (4 096-row) edges, with exact
ties, duplicate rows and every label layout from two labels to n - 1; agreement with sklearn; bit-identical reruns and
batch splits; the memory refusal; and the cell-type and modality silhouettes of a trained model's joint embedding."""
import ctypes as C
import os

import numpy as np
import pytest
from sklearn.metrics import silhouette_samples as sk_samples
from sklearn.metrics import silhouette_score as sk_score

from tests import silhouette_oracle as S

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'mmdma.npz')
EDGES = [63, 64, 65, 127, 128, 129, 4095, 4096, 4097, 8191, 8192, 8193, 69631, 69632, 69633]


def _rows(kind, n, L, rng):
    if kind == 'normal':
        return rng.standard_normal((n, L)).astype(np.float32)
    if kind == 'grid':                                   # exact ties everywhere
        return rng.integers(-2, 3, (n, L)).astype(np.float32)
    if kind == 'duplicates':                             # each row repeated, in scattered places: zero distances
        base = rng.standard_normal((max(1, n // 3), L)).astype(np.float32)
        return base[rng.integers(0, base.shape[0], n)]
    raise ValueError(kind)


def _offsets(layout, n, rng):
    """int64 label offsets [C + 1] of rows sorted by label."""
    if layout == 'two':
        cuts = [n // 2]
    elif layout == 'one_vs_rest':
        cuts = [1]
    elif layout == 'random20':
        cuts = sorted(rng.choice(np.arange(1, n), min(19, n - 2), replace=False).tolist())
    elif layout == 'n_minus_1':                          # one label of two rows, every other row alone
        cuts = list(range(2, n))
    elif layout == 'edges':                              # segments ending one row either side of tile and chunk edges
        cuts = [e for e in EDGES if 0 < e < n] or [1]
    else:
        raise ValueError(layout)
    return np.array([0, *cuts, n], np.int64)


def _sums(x, off, batch_bytes=1 << 30):
    from jamie_b200.evaluation import DeviceSilhouette
    return DeviceSilhouette.sums(np.ascontiguousarray(x, np.float32), off, batch_bytes, None)


def _checked_rows(n, off, rng):
    """Every row for small n; else 400 random rows, the rows at tile / chunk edges and, for up to 100 labels, at each
    label's ends."""
    if n <= 1000:
        return np.arange(n)
    ends = off.tolist() if len(off) <= 100 else []
    near = [r for o in ends + EDGES for r in (o - 1, o) if 0 <= r < n]
    return np.unique(np.concatenate([rng.choice(n, 400, replace=False), near, [0, n - 1]]))


# n in {3, 63, 64, 65, 4095, 4096, 4097, 70000}, each with an L in {1, 2, 32, 33, 100}
SHAPES = [(3, 1), (63, 33), (64, 2), (65, 100), (4095, 32), (4096, 1), (4097, 33), (70000, 32), (4097, 100), (70000, 2)]


@pytest.mark.parametrize('n,L', SHAPES)
@pytest.mark.parametrize('layout', ['two', 'one_vs_rest', 'random20', 'n_minus_1', 'edges'])
@pytest.mark.parametrize('kind', ['normal', 'grid', 'duplicates'])
def test_sums_equal_the_reference(n, L, layout, kind):
    rng = np.random.default_rng(n * 31 + L)
    x = _rows(kind, n, L, rng)
    off = _offsets(layout, n, rng)
    intra, inter = _sums(x, off)
    codes = np.repeat(np.arange(len(off) - 1), np.diff(off))
    rows = _checked_rows(n, off, rng)
    oi, oe = S.sums(x, codes, rows)
    np.testing.assert_allclose(intra[rows], oi, rtol=1e-12, atol=0)
    np.testing.assert_allclose(inter[rows], oe, rtol=1e-12, atol=0)
    assert np.all(np.isfinite(intra)) and np.all(np.isfinite(inter)) and np.all(intra >= 0) and np.all(inter >= 0)


def test_silhouette_samples_matches_sklearn():
    from jamie_b200.evaluation import silhouette_samples, silhouette_score
    rng = np.random.default_rng(1)
    centres = rng.standard_normal((20, 16)) * 3
    types = rng.integers(0, 20, 5000)
    X = centres[types] + rng.standard_normal((5000, 16))
    X64 = X.astype(np.float32).astype(np.float64)        # no duplicate rows; float32 rows, as the device reads them
    for labels in (types, rng.integers(0, 2, 5000), np.array([f'type {t % 7}' for t in types])):
        got = silhouette_samples(X64, labels)
        np.testing.assert_allclose(got, sk_samples(X64, labels), rtol=0, atol=1e-12)
        np.testing.assert_allclose(got, S.silhouette_samples(X64, labels), rtol=0, atol=1e-12)
        X32 = X.astype(np.float32)                       # sklearn's float32 path differs by about 2e-7
        np.testing.assert_allclose(silhouette_samples(X32, labels), sk_samples(X32, labels), rtol=0, atol=1e-6)
        assert abs(silhouette_score(X64, labels) - sk_score(X64, labels)) < 1e-12
        assert abs(silhouette_score(X64, labels, sample_size=1000, random_state=3)
                   - sk_score(X64, labels, sample_size=1000, random_state=3)) < 1e-12


def test_bit_identical_reruns_and_batches():
    rng = np.random.default_rng(2)
    n = 5000
    x = np.concatenate([_rows('normal', 3000, 33, rng), _rows('grid', 2000, 33, rng)])
    off = _offsets('edges', n, rng)
    off = np.unique(np.concatenate([off, _offsets('random20', n, rng)]))
    chunk_labels = [np.searchsorted(off, min(n, c0 + 4096) - 1, side='right') - np.searchsorted(off, c0, side='right') + 1
                    for c0 in range(0, n, 4096)]
    row_b = 8 * sum(chunk_labels) + 16                     # one query row's slots and outputs
    ref = _sums(x, off)
    for bb in (1 << 30, 1, 100 * row_b):                  # one batch; one row a batch; 64 rows a batch
        intra, inter = _sums(x, off, batch_bytes=bb)
        np.testing.assert_array_equal(intra, ref[0])
        np.testing.assert_array_equal(inter, ref[1])
    np.testing.assert_array_equal(_sums(x, off)[0], ref[0])


def test_refuses_a_problem_larger_than_free_memory():
    import torch
    from jamie_b200 import _lib
    from jamie_b200.evaluation import silhouette_samples
    lib = _lib.load()
    p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    free0 = torch.cuda.mem_get_info()[0]
    z = np.zeros(16, np.float32)
    out = np.zeros(4)
    n = (1 << 31) - 1
    rc = lib.jb_silhouette(p(z), n, 1 << 20, p(np.array([0, 1, n], np.int64)), 2, 1 << 30, 0, p(out), p(out))   # 9 PB
    assert rc != 0
    msg = lib.jb_last_error().decode()
    assert 'GB' in msg and 'free' in msg, msg
    for off, nl in (([1, 2, 4], 2), ([0, 2, 2, 4], 3), ([0, 4], 1), ([0, 1, 3], 2)):   # bad offsets, 1 label, sum != n
        rc = lib.jb_silhouette(p(z), 4, 4, p(np.array(off, np.int64)), nl, 1 << 30, 0, p(out), p(out))
        assert rc != 0 and 'label' in lib.jb_last_error().decode()
    assert abs(torch.cuda.mem_get_info()[0] - free0) < (64 << 20)
    rng = np.random.default_rng(0)
    x, labels = _rows('normal', 50, 4, rng), rng.integers(0, 3, 50)
    np.testing.assert_allclose(silhouette_samples(x, labels), S.silhouette_samples(x, labels), rtol=0, atol=1e-12)


def test_end_to_end_joint_embedding():
    from jamie import JAMIE
    from jamie.evaluation import silhouette_samples, silhouette_score
    g = np.load(GOLD)
    data = [g['data1'].astype(np.float32), g['data2'].astype(np.float32)]
    np.random.seed(1)
    jm = JAMIE(output_dim=8, batch_size=64, pca_dim=[20, 16], epoch_DNN=20, min_epochs=1, use_f_tilde=False, manual_seed=5)
    try:
        emb = jm.fit_transform(dataset=[x.copy() for x in data], P=np.eye(data[0].shape[0]))
    finally:
        jm.engine.close()
    joint = np.concatenate(emb)
    types = np.concatenate([g['type1'], g['type2']])
    modality = np.repeat([0, 1], [len(emb[0]), len(emb[1])])
    for labels in (types, modality):
        got = silhouette_samples(joint, labels)
        assert got.shape == (joint.shape[0],) and np.all(np.abs(got) <= 1)
        np.testing.assert_allclose(got, sk_samples(joint, labels), rtol=0, atol=1e-6)
        np.testing.assert_allclose(got, S.silhouette_samples(joint, labels), rtol=0, atol=1e-12)
        assert abs(silhouette_score(joint, labels) - float(np.mean(got))) == 0
