"""Randomized PCA fit (JAMIE(pca_fit='randomized'), jamie_b200/pca_fit.py randomized_fit_transform): GPU phases against
the same algorithm on the host.

  python tools/pca_bench.py [--quick] [--out FILE.md]

Shapes: dense 4 301 x 85 596 (DM_rep4's width) and sparse 100 000 x 60 000 at 5 % density, k = 512 (--quick: small
shapes, for a rehearsal). GPU phases: operand upload (create), column statistics, operand products, QR, and the rest
(downloads, the host SVD of the l x (n or d) matrix B, U = Q U_hat). Host: sklearn.utils.extmath._randomized_svd on
_implicit_column_offset(X, mean), the call PCA(svd_solver='randomized') makes; for the sparse shape only one host product
is timed, on its first 10 000 rows, and the full fit is extrapolated (2 n_iter + 2 products), as scipy's
single-threaded sparse products make the whole fit take tens of minutes. The Gram route (pca_fit='gpu') needs a d x d matrix (58 GB at d = 85 596, 29 GB at
d = 60 000) and a host eigensolve of it: not run at these shapes.
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU
HOST_ROWS = 10000          # sparse host arm: rows of the one timed product


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def dense_data(n, d, seed):
    rng = np.random.default_rng(seed)
    r = 64
    lat = rng.standard_normal((n, r), dtype=np.float32) * np.linspace(3.0, 0.3, r, dtype=np.float32)
    X = lat @ rng.standard_normal((r, d), dtype=np.float32)
    X += 0.1 * rng.standard_normal((n, d), dtype=np.float32)
    X += 2.0 * rng.standard_normal(d, dtype=np.float32)
    return X


def sparse_data(n, d, density, seed):
    """CSR with about density * n * d stored entries: log-normal-ish counts at random positions (an expression matrix)"""
    rng = np.random.default_rng(seed)
    per_row = rng.binomial(d, density, size=n)
    indptr = np.zeros(n + 1, np.int64)
    np.cumsum(per_row, out=indptr[1:])
    nnz = int(indptr[-1])
    idx = np.empty(nnz, np.int32)
    for r0 in range(0, n, 4096):   # sorted distinct columns per row
        for r in range(r0, min(n, r0 + 4096)):
            idx[indptr[r]:indptr[r + 1]] = np.sort(rng.choice(d, per_row[r], replace=False))
    val = np.exp(rng.standard_normal(nnz, dtype=np.float32)).astype(np.float32)
    return sp.csr_matrix((val, idx, indptr), shape=(n, d))


class Timed:
    """DeviceOperator with per-phase device-synchronised timers"""

    def __init__(self, base):
        self.base, self.t, self.n_apply = base, {}, 0

    def __call__(self, X, device):
        import torch
        t0 = time.perf_counter()
        self.op = self.base(X, device)
        torch.cuda.synchronize()
        self.t['upload'] = time.perf_counter() - t0
        return self

    def _time(self, phase, fn, *a):
        import torch
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn(*a)
        torch.cuda.synchronize()
        self.t[phase] = self.t.get(phase, 0.0) + time.perf_counter() - t0
        return out

    def stats(self):
        return self._time('stats', self.op.stats)

    def upload(self, a):
        return self.op.upload(a)

    def apply(self, trans, B):
        self.n_apply += 1
        self.l = B.shape[1]
        return self._time('products', self.op.apply, trans, B)

    def orth(self, Y):
        return self._time('qr', self.op.orth, Y)

    def download(self, Y):
        return self._time('rest', self.op.download, Y)

    def close(self):
        self.op.close()


def gpu_fit(X, k, seed=0):
    from jamie_b200 import pca_fit
    import torch
    pca_fit.randomized_fit_transform(X[:64] if not sp.issparse(X) else X[:64], min(k, 8), seed, 0)   # warm-up: module load, cuSOLVER
    torch.cuda.synchronize()
    tm = Timed(pca_fit.DeviceOperator)
    t0 = time.perf_counter()
    pca, sample = pca_fit.randomized_fit_transform(X, k, seed, 0, operator=tm)
    total = time.perf_counter() - t0
    tm.t['rest'] = total - sum(v for p, v in tm.t.items() if p != 'rest')
    return pca, total, tm


def host_fit(X, k, seed, one_product):
    from sklearn.decomposition._pca import _implicit_column_offset
    from sklearn.utils.extmath import _randomized_svd
    mean = np.asarray(X.mean(axis=0), np.float64).ravel().astype(X.dtype)
    A = _implicit_column_offset(X, mean)
    n, d = X.shape
    l = min(k + 10, n, d)
    n_iter = 7 if k < 0.1 * min(n, d) else 4
    if one_product:   # Xc @ Omega on the first HOST_ROWS rows, scaled to all n rows
        rows = min(n, HOST_ROWS)
        Om = np.random.default_rng(seed).standard_normal((d, l), dtype=np.float32)
        t0 = time.perf_counter()
        _implicit_column_offset(X[:rows], mean) @ Om
        t1 = (time.perf_counter() - t0) * n / rows
        return None, t1 * (2 * n_iter + 2), t1
    t0 = time.perf_counter()
    _randomized_svd(A, k, n_oversamples=10, n_iter='auto', flip_sign=False, random_state=seed)
    return None, time.perf_counter() - t0, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--quick', action='store_true', help='small shapes (rehearsal)')
    ap.add_argument('--out', default=None, help='write the markdown table here')
    ap.add_argument('--no-host', action='store_true')
    ap.add_argument('--shape', choices=('dense', 'sparse', 'both'), default='both')
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('pca_bench needs a CUDA device: there is nothing to measure without one')
    shapes = [('dense', 4301, 85596, 1.0, 512), ('sparse', 100000, 60000, 0.05, 512)]
    if args.quick:
        shapes = [('dense', 300, 2000, 1.0, 32), ('sparse', 3000, 1500, 0.05, 32)]
    shapes = [s for s in shapes if args.shape in ('both', s[0])]
    dev = card()
    rows = []
    for kind, n, d, dens, k in shapes:
        t0 = time.perf_counter()
        X = dense_data(n, d, 0) if kind == 'dense' else sparse_data(n, d, dens, 0)
        gen = time.perf_counter() - t0
        pca, total, tm = gpu_fit(X, k)
        l = tm.l
        nnz = X.nnz if kind == 'sparse' else n * d
        per_apply = tm.t['products'] / tm.n_apply
        row = dict(kind=kind, n=n, d=d, nnz=nnz, k=k, l=l, total=total, gen=gen, n_apply=tm.n_apply, **tm.t)
        if kind == 'sparse':
            # per product: the nonzeros (int32 index + fp32 value), B read once, Y written once; and the row gathers
            # (l fp32 per nonzero) as they would cost if none hit in L2
            comp = nnz * 8 + (n + d) * l * 4
            row['compulsory_GBps'] = comp / per_apply / 1e9
            row['gather_GBps'] = (nnz * l * 4) / per_apply / 1e9
        else:
            row['tflops'] = 2.0 * n * d * l / per_apply / 1e12
        if not args.no_host:
            _, host_t, one = host_fit(X, k, 0, one_product=(kind == 'sparse' and not args.quick))
            row['host'] = host_t
            row['host_one_product'] = one
        rows.append(row)
        print(row, flush=True)
        del X
    lines = [f'Card: {dev} (nvidia-smi name, power limit), read in the same run.', '',
             '| input | n x d | nnz | k (l) | GPU fit s | upload | stats | products (count) | QR | host SVD + rest | host fit s |',
             '|---|---|---|---|---|---|---|---|---|---|---|']
    for r in rows:
        host = 'not measured'
        if 'host' in r:
            host = f"{r['host']:.1f}" if r['host_one_product'] is None else \
                f"~{r['host']:.0f} (estimate: {r['n_apply']} x one product, {r['host_one_product']:.1f} s scaled from {HOST_ROWS} rows)"
        lines.append(f"| {r['kind']} | {r['n']} x {r['d']} | {r['nnz']:.3g} | {r['k']} ({r['l']}) | {r['total']:.2f} | "
                     f"{r['upload']:.2f} | {r['stats']:.3f} | {r['products']:.2f} ({r['n_apply']}) | {r['qr']:.2f} | "
                     f"{r['rest']:.2f} | {host} |")
    lines.append('')
    for r in rows:
        per = r['products'] / r['n_apply']
        if r['kind'] == 'sparse':
            lines.append(f"- sparse products: {per * 1e3:.1f} ms each; compulsory bytes (nonzeros + B + Y) "
                         f"{r['compulsory_GBps']:.0f} GB/s = {r['compulsory_GBps'] * 1e9 / HBM_BYTES_PER_S:.1%} of 7.7 TB/s; "
                         f"row gathers counted as if none hit in L2: {r['gather_GBps']:.0f} GB/s")
        else:
            lines.append(f"- dense products: {per * 1e3:.1f} ms each, {r['tflops']:.1f} TFLOP/s counting 2 n d l per product "
                         f"(3xTF32 issues three TF32 products for each)")
    text = '\n'.join(lines) + '\n'
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text)


if __name__ == '__main__':
    main()
