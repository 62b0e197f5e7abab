"""What SISA slicing (Sisa.slices = R) costs and saves: learn time, unlearn time per kind of request, trained
interactions and accuracy after learn, for R in {1, 2, 4, 8}.

    python tools/prof_slices.py [--reps 3] [--out result.json] [--skip-c3]

Two shapes, uniform grouping, batch 30 000, E = 50, epoch_eval 'final':
  * ml1m: synth.ml_like (6040 users x 3416 items, 897 k training rows), K = 5, d = 16;
  * C3: 138 493 users x 26 744 items, 20 M training rows (users sorted, items uniform, ratings 1..5) and 2 M test
    rows, K = 8, d = 64.
Unlearn requests: one deleted user of shard 0 whose slice is the first, the middle (R // 2) or the last; the 2 %
`rand` user set (np.random.seed(0), as InsParam draws it); 2 % of the training rows as `inter` pairs.  Each learn and
each unlearn runs once to warm up and `reps` more times; the median host time around the call, ended by a device
synchronise, is reported (the ingest of the retained data is not included).  RMSE / NDCG@10 / HR@10 are the learn
pass's final evaluation.  The card name and power limit are printed with the numbers.
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
from ultrare_b200 import synth                                               # noqa: E402
from ultrare_b200.config import routed_users                                 # noqa: E402
from ultrare_b200.method.sisa import Sisa, stage_epochs                      # noqa: E402
from ultrare_b200.read import loadData, readRatingDevice                     # noqa: E402

SLICES = (1, 2, 4, 8)


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ''
    return q or torch.cuda.get_device_name(0) + ', power limit unknown'


def timed(fn, reps):
    fn()                                   # warm-up
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t) * 1e3)
    return float(np.median(ts)), out


def scenario(name, train, test, U, I, K, d, E, reps):
    class P:
        n_user, n_item, k, lam, seed, lr, lr_decay, momentum, batch = U, I, d, 0.1, 42, 0.001, 0.95, 0.9, 30000
    P.epochs = E
    tr = pd.DataFrame({0: train[0], 1: train[1], 2: train[2]})
    te = pd.DataFrame({0: test[0], 1: test[1], 2: test[2]})
    n = len(tr)
    np.random.seed(0)
    rand_users = np.random.choice(U, int(0.02 * U), replace=False)
    np.random.seed(0)
    rows = np.sort(np.random.choice(n, int(0.02 * n), replace=False))
    pairs = np.stack([train[0][rows], train[1][rows]], 1).astype(np.int64)
    _, groups, _ = readRatingDevice(tr, U, 5, [], [], K, [], 'r', device='cuda')
    tds, _, ttot = readRatingDevice(te, U, 5, [], [], K, groups, 'r', device='cuda')
    test_dl = [loadData(x, 30000, 1, False) for x in tds]
    test_data = loadData(ttot, 30000, 1, False)
    res = []
    for R in SLICES:
        ds, _, _ = readRatingDevice(tr, U, 5, [], [], K, groups, 'r', device='cuda', n_slice=R)
        train_dl = [loadData(x, 30000, 1, True) for x in ds]

        def learn():
            s = Sisa(P, 'mf', K, groups)
            s.epoch_eval, s.slices = 'final', R
            s.learn(train_dl, test_dl, test_data, 0, '')
            return s
        learn_ms, s = timed(learn, reps)
        row = dict(R=R, stage_epochs=stage_epochs(E, R), learn_ms=learn_ms,
                   learn_trained=s.timing['trained_interactions'] if R > 1 else sum(len(x) for x in ds) * E,
                   rmse=s.final_log['total_rmse'], ndcg=s.final_log['total_ndcg'], hr=s.final_log['total_hr'])
        models = s.model_list
        w = models[0].user_mat.weight
        g0 = groups[0]
        one = {k: [int(g0[-(-a * len(g0) // R)])] for k, a in
               (('one_first', 0), ('one_middle', R // 2), ('one_last', R - 1))}
        kinds = dict(one, rand=(list(rand_users), []), inter=([], pairs))
        for kind, req in kinds.items():
            du, dr = (req, []) if kind.startswith('one') else req
            dds, _, _ = readRatingDevice(tr, U, 5, du, dr, K, groups, 'r', device='cuda', n_slice=R)
            dl = [loadData(x, 30000, 1, True) for x in dds]
            users = routed_users(du, dr)

            def unlearn():
                for m in models:
                    m.user_mat.weight = w
                s2 = Sisa(P, 'mf', K, groups)
                s2.epoch_eval, s2.slices = 'final', R
                s2.unlearn(models, dl, test_dl, test_data, users, 0, '')
                return s2
            ms, s2 = timed(unlearn, reps)
            trained = s2.timing['trained_interactions'] if R > 1 else \
                sum(len(dds[g]) for g in s2.retrain_gid) * E
            row[kind] = dict(ms=ms, trained=trained, shards=len(s2.retrain_gid),
                             first=s2.first_slice.tolist() if R > 1 else None)
        for m in models:
            m.user_mat.weight = w
        res.append(row)
        print(f"{name} R={R} (e'={row['stage_epochs']}): learn {learn_ms:.0f} ms, {row['learn_trained']:.3e} trained | "
              f"RMSE {row['rmse']:.4f} NDCG@10 {row['ndcg']:.4f} HR@10 {row['hr']:.4f} | unlearn ms (trained): " +
              ", ".join(f"{k} {row[k]['ms']:.0f} ({row[k]['trained']:.2e})" for k in kinds), flush=True)
        del s, models, w, train_dl, ds
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default=None)
    ap.add_argument('--skip-c3', action='store_true')
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.zeros(1, device='cuda')
    res = dict(card=card())
    print('card:', res['card'], flush=True)
    train, test = synth.ml_like()
    res['ml1m'] = scenario('ml1m', train, test, 6040, 3416, 5, 16, 50, a.reps)
    if not a.skip_c3:
        rng = np.random.default_rng(1)
        U, I = 138_493, 26_744
        mk = lambda n: (np.sort(rng.integers(0, U, n)), rng.integers(0, I, n), rng.integers(1, 6, n).astype(float))
        train, test = mk(20_000_000), mk(2_000_000)
        res['c3'] = scenario('c3', train, test, U, I, 8, 64, 50, max(1, a.reps - 1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
