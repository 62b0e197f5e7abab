"""Cost of the 'rating-ot' grouping: the sparse cost and centroid kernels, one outer iteration, the whole grouping.

    python tools/prof_rating_ot.py [--reps 50] [--out result.json]

Shapes: ml1m (synth.ml_like: 6 040 x 3 416, 897 k ratings) and C3 (138 493 x 26 744, 20 M ratings drawn uniformly, one
user-sorted file), each at k in {5, 8, 64}.  With CUDA events, after warm-up: ure_sparse_cost (with the inertia) and
ure_sparse_centroid_sums, with the bytes each must move (the CSR / CSC arrays, one kpad-wide Ct row gathered per
nonzero, the label gathered per nonzero, the outputs) over the time.  The ml1m working set stays in L2 between
repetitions; C3's (~240 MB of CSR + CSC) does not.  With the host clock: the device set-up (upload of the records and
the three radix sorts of kernels.sparse_orders), one outer iteration (ot_cluster_sparse_device with max_iters=1, set-up
included), the whole grouping (default options), and the host baseline -- SciPy's sparse X @ C.T plus the centroid sums
as a sparse one-hot product.  The card name and power limit are printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ultrare_b200 import kernels as kn, synth                       # noqa: E402
from ultrare_b200.method.utils import ot_cluster_sparse_device, sparse_records   # noqa: E402


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ''
    return q or torch.cuda.get_device_name(0) + ', power limit unknown'


def events_ms(fn, reps):
    for _ in range(3):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def host_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3 / reps


def shape(name, X, ks, reps):
    dev = torch.device('cuda', 0)
    n, n_item = X.shape
    nnz = X.nnz
    rec = sparse_records(X)
    setup = host_ms(lambda: kn.sparse_orders(kn.upload_table(rec, dev), n, n_item), 3)
    csr, csc = kn.sparse_orders(kn.upload_table(rec, dev), n, n_item)
    out = dict(users=n, items=n_item, nnz=nnz, setup_ms=setup, k={})
    print(f"{name}: {n} x {n_item}, {nnz} ratings | set-up (upload + orders) {setup:.2f} ms", flush=True)
    rng = np.random.default_rng(0)
    for k in ks:
        kp = kn.kpad_for(k)
        np.random.seed(0)
        c0 = X[np.random.choice(n, size=k, replace=False)].toarray()
        Ct = np.zeros((n_item, kp), dtype=np.float32)
        Ct[:, :k] = c0.T
        Ctd = kn.upload_array(Ct, dev)
        cn = kn.upload_array(np.square(c0.astype(np.float64)).sum(axis=1), dev)
        label = torch.tensor(rng.integers(0, k, n).astype(np.int32), device=dev)
        cost = events_ms(lambda: kn.sparse_cost(csr, Ctd, cn, k, want_inertia=True), reps)
        cen = events_ms(lambda: kn.sparse_centroid_sums(csc, label, k), reps)
        cost_b = 8 * (n + 1) + 8 * nnz + 4 * kp * nnz + 4 * kp * n + 8 * k
        cen_b = 8 * (n_item + 1) + 12 * nnz + 8 * kp * n_item + 4 * n
        one = host_ms(lambda: ot_cluster_sparse_device(X, k, max_iters=1, centroid0=c0), 3)
        np.random.seed(0)
        t = time.perf_counter()
        _, lab, _, iters = ot_cluster_sparse_device(X, k)
        whole = (time.perf_counter() - t) * 1e3
        Xh = X.tocsr()
        L = sp.csr_matrix((np.ones(n, dtype=np.float64), (lab, np.arange(n))), shape=(k, n))

        def host():
            Xh @ c0.T
            L @ Xh
        hb = host_ms(host, 3)
        r = dict(kpad=kp, cost_ms=cost, cost_GBps=cost_b / cost / 1e6, centroid_ms=cen, centroid_GBps=cen_b / cen / 1e6,
                 one_iteration_ms=one, grouping_ms=whole, outer_iterations=iters, host_baseline_ms=hb,
                 sizes=np.bincount(lab, minlength=k).tolist()[:8])
        out['k'][k] = r
        print(f"  k={k} (kpad {kp}): cost {cost:.3f} ms ({r['cost_GBps']:.0f} GB/s) | centroid sums {cen:.3f} ms "
              f"({r['centroid_GBps']:.0f} GB/s) | one iteration {one:.1f} ms | grouping {whole:.1f} ms ({iters} iterations)"
              f" | host X @ C.T + sums {hb:.1f} ms", flush=True)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--reps', type=int, default=50)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.zeros(1, device='cuda')
    res = dict(card=card())
    print('card:', res['card'], flush=True)
    (u, i, r), _ = synth.ml_like()
    X = sp.coo_matrix(((r / 5).astype(np.float32), (u, i)), shape=(6040, 3416), dtype=np.float32).tocsr()
    res['ml1m'] = shape('ml1m', X, (5, 8, 64), a.reps)
    rng = np.random.default_rng(1)
    n, U, I = 20_000_000, 138_493, 26_744
    X = sp.coo_matrix(((rng.integers(1, 6, n) / 5).astype(np.float32), (np.sort(rng.integers(0, U, n)),
                                                                         rng.integers(0, I, n))),
                      shape=(U, I), dtype=np.float32).tocsr()
    res['c3'] = shape('c3', X, (5, 8, 64), a.reps)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
