"""Cost of interaction-level unlearning (deleted (user, item) ratings) on the device ingest, and one ml1m unlearn pass.

    python tools/prof_unlearn_inter.py [--reps 50] [--epochs 10] [--out result.json]

At two sizes -- ml1m (synth.ml_like: 897 k rows, 2 % of them deleted) and a C3-sized table (20 M rows sorted by user,
138 493 users x 26 744 items, 1 % deleted) -- it times with CUDA events:
  * the partition (ure_partition_interactions) without deletion lists and with them (ure_partition_interactions_del),
  * the deleted-item CSR build (kernels.deletion_lists: upload of the pairs, id checks, ure_seen_lists), end to end,
and with the host clock the host readRating with and without the pair filter.  The ml1m table (21 MB) stays in L2
between repetitions; the 20 M-row table (480 MB) does not.  Then one ml1m Sisa.unlearn pass (K = 5, epoch_eval
'none') after an `inter` draw (2 % of the rows: every shard is routed) beside a `rand` draw (2 % of the users).
The card name and power limit are printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import pandas as pd
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ultrare_b200 import kernels as kn, synth                       # noqa: E402
from ultrare_b200.read import RatingData, loadData, readRating, readRatingDevice   # noqa: E402


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


def ingest(name, u, i, r, n_user, frac, reps, K=5):
    dev = torch.device('cuda', 0)
    n = len(u)
    rng = np.random.default_rng(0)
    rows = np.sort(rng.choice(n, int(frac * n), replace=False))
    pairs = np.stack([u[rows], i[rows]], 1).astype(np.int64)
    n_map = max(n_user, int(u.max()) + 1)
    owner = np.full(n_map, -1, dtype=np.int32)
    owner[:n_user] = rng.permutation(n_user) % K
    table = kn.upload_table(np.stack([u.astype(np.float64), i.astype(np.float64), r.astype(np.float64)]), dev)
    own = kn.upload_array(owner, dev)
    lists = kn.deletion_lists(pairs, n_map, dev)
    plain = events_ms(lambda: kn.partition_interactions(table, 5, own, None, K), reps)
    listed = events_ms(lambda: kn.partition_interactions(table, 5, own, None, K, del_lists=lists), reps)
    build = host_ms(lambda: kn.deletion_lists(pairs, n_map, dev), max(3, reps // 5))
    _, o0 = kn.partition_interactions(table, 5, own, None, K)
    _, o1 = kn.partition_interactions(table, 5, own, None, K, del_lists=lists)
    dropped = int(o0[-1]) - int(o1[-1])
    df = pd.DataFrame({0: u, 1: i, 2: r})
    hreps = 3 if n > 5_000_000 else 10
    h_plain = host_ms(lambda: readRating(df, n_user, 5, [], [], K), hreps)
    h_pairs = host_ms(lambda: readRating(df, n_user, 5, [], pairs, K), hreps)
    out = dict(size=name, rows=n, pairs=len(pairs), rows_dropped=dropped, partition_ms=plain,
               partition_del_ms=listed, partition_del_extra_ms=listed - plain, csr_build_ms=build,
               host_readRating_ms=h_plain, host_readRating_pairs_ms=h_pairs,
               partition_GBps=n * 24 / plain / 1e6, partition_del_GBps=n * 24 / listed / 1e6)
    print(f"{name}: {n} rows, {len(pairs)} pairs ({dropped} rows dropped) | partition {plain:.3f} ms, with lists "
          f"{listed:.3f} ms (+{listed - plain:.3f}) | CSR build {build:.3f} ms | host readRating {h_plain:.1f} ms, "
          f"with pairs {h_pairs:.1f} ms", flush=True)
    return out


def unlearn_pass(epochs):
    from ultrare_b200.method.sisa import Sisa
    U, I, K, B = 6040, 3416, 5, 30000
    train, test = synth.ml_like()
    tr = pd.DataFrame({0: train[0], 1: train[1], 2: train[2]})
    te = pd.DataFrame({0: test[0], 1: test[1], 2: test[2]})
    trr, groups = readRating(tr, U, 5, [], [], K, [], 'a')
    ter, _ = readRating(te, U, 5, [], [], K, groups)

    class P:
        n_user, n_item, k, lam, seed, lr, lr_decay, momentum, batch = U, I, 16, 0.1, 42, 0.001, 0.95, 0.9, B
    P.epochs = epochs
    test_dl = [loadData(RatingData(a), B, 1, False) for a in ter]
    test_data = loadData(RatingData(np.hstack(ter)), B, 1, False)
    s = Sisa(P, 'mf', K, groups)
    s.epoch_eval = 'none'
    before = s.learn([loadData(RatingData(a), B, 1, True) for a in trr], test_dl, test_data, 0, '')
    w = before[0].user_mat.weight
    rng = np.random.RandomState(0)
    rows = np.sort(rng.choice(len(train[0]), int(0.02 * len(train[0])), replace=False))
    pairs = np.stack([train[0][rows], train[1][rows]], 1).astype(np.int64)
    del_user = np.random.RandomState(0).choice(U, int(0.02 * U), replace=False)
    out = {}
    for kind, du, dr in (('rand', del_user, []), ('inter', sorted(set(pairs[:, 0].tolist())), pairs)):
        for m in before:
            m.user_mat.weight = w
        torch.cuda.synchronize()
        t = time.perf_counter()
        ds, _, _ = readRatingDevice(tr, U, 5, list(du) if kind == 'rand' else [], dr, K, groups, 'r')
        s2 = Sisa(P, 'mf', K, groups)
        s2.epoch_eval = 'none'
        s2.unlearn(before, [loadData(d, B, 1, True) for d in ds], test_dl, test_data, du, 0, '')
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t) * 1e3
        out[kind] = dict(unlearn_ms=ms, retrained=sorted(s2.retrain_gid), rows_trained=sum(len(d) for d in ds))
        print(f"ml1m unlearn ({kind}, {epochs} epochs, ingest included): {ms:.0f} ms, shards {sorted(s2.retrain_gid)}, "
              f"{out[kind]['rows_trained']} rows", flush=True)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--reps', type=int, default=50)
    ap.add_argument('--epochs', type=int, default=10)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.zeros(1, device='cuda')
    res = dict(card=card())
    print('card:', res['card'], flush=True)
    train, _ = synth.ml_like()
    res['ml1m'] = ingest('ml1m', train[0], train[1], train[2], 6040, 0.02, a.reps)
    rng = np.random.default_rng(1)
    n, U, I = 20_000_000, 138_493, 26_744
    res['c3'] = ingest('c3', np.sort(rng.integers(0, U, n)), rng.integers(0, I, n), rng.integers(1, 6, n).astype(float),
                       U, 0.01, a.reps)
    res['unlearn'] = unlearn_pass(a.epochs)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
