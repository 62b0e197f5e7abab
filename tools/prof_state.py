"""What a saved SISA state costs: save, load, one deletion request from the loaded state against the same unlearn in
the process that learned, and the state's size on disk, at R = 1 and 8.

    python tools/prof_state.py [--out result.json] [--skip-c3] [--dir DIR]

Two shapes, uniform grouping, batch 30 000, E = 50, epoch_eval 'final', combine 'mean', data written as CSV under
--dir (default: a temporary directory, removed at the end):
  * ml1m: synth.ml_like (6040 users x 3416 items, 897 k training rows), K = 5, d = 16;
  * C3: 138 493 users x 26 744 items, 20 M training rows and 2 M test rows (as tools/prof_slices.py), K = 8, d = 64.
The request is the 2 % `rand` user set (np.random.seed(0), as InsParam draws it).  Times are host times ended by a
device synchronise, one run each after a learn that warms every kernel: save_state (device-to-host copy and the files),
load_state (module caches cleared, as in a new process), the retained-data read (CSV parse and device ingest), the
request's unlearn (apply_request on the read data) and the in-process unlearn of the same request on the learned
model.  The card name and power limit are printed with the numbers.
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from prof_slices import card                                                 # noqa: E402
from ultrare_b200 import kernels as kn                                       # noqa: E402
from ultrare_b200 import synth                                               # noqa: E402
from ultrare_b200.method import sisa as msisa                                # noqa: E402
from ultrare_b200.method import sisa_state as st                            # noqa: E402
from ultrare_b200.method.sisa import Sisa                                    # noqa: E402

SLICES = (1, 8)


def clock(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, out


def du(path):
    return sum(os.path.getsize(os.path.join(path, n)) for n in os.listdir(path))


def scenario(name, train, test, U, I, K, d, E, root):
    class P:
        n_user, n_item, k, lam, seed, lr, lr_decay, momentum, batch = U, I, d, 0.1, 42, 0.001, 0.95, 0.9, 30000
    P.epochs = E
    paths = {p: os.path.join(root, name, p + '.csv') for p in ('train', 'test')}
    synth.write_csv(paths['train'], train)
    synth.write_csv(paths['test'], test)
    src = dict(dataset=name, train_file=paths['train'], test_file=paths['test'], max_rating=5, grouping='uniform',
               group_index=[])
    np.random.seed(0)
    users = np.random.choice(U, int(0.02 * U), replace=False)
    res = []
    for R in SLICES:
        tl, sl, total, idx = st.read_retained(src, U, K, R, 30000, [], [])
        s = Sisa(P, 'mf', K, idx)
        s.source, s.slices, s.epoch_eval = dict(src), R, 'final'
        learn_ms, _ = clock(lambda: s.learn(tl, sl, total, 0, ''))
        sdir = os.path.join(root, name, f'state_R{R}')
        save_ms, _ = clock(lambda: s.save_state(sdir))
        msisa._OWNER_CACHE.clear()
        msisa._EVAL_ROWS.clear()
        kn._PLAN_HINTS.clear()
        load_ms, L = clock(lambda: Sisa.load_state(sdir))
        read_ms, data = clock(lambda: L.retained_data(users, ()))
        req_ms, _ = clock(lambda: L.apply_request(users, (), *data))
        s2 = Sisa(P, 'mf', K, idx)
        s2.slices, s2.epoch_eval = R, 'final'
        inproc_ms, _ = clock(lambda: s2.unlearn(s.model_list, *data, list(users), 0, ''))
        a, b = L.model_list[0].user_mat.weight.data, s2.model_list[0].user_mat.weight.data
        same = bool(torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(a.nan_to_num(), b.nan_to_num()))
        nan_rows = int(torch.isnan(a).any(1).sum())
        ck = [sum(os.path.getsize(os.path.join(sdir, f'ckpt{g}_{r}_{m}.npy')) for r in range(R) for m in 'PQ')
              if R > 1 else 0 for g in range(K)]
        row = dict(R=R, learn_ms=learn_ms, save_ms=save_ms, load_ms=load_ms, read_retained_ms=read_ms,
                   request_unlearn_ms=req_ms, inprocess_unlearn_ms=inproc_ms, merged_equal=same, merged_nan_rows=nan_rows,
                   state_bytes=du(sdir), ckpt_bytes_per_shard_max=max(ck), shards_retrained=len(L.retrain_gid))
        res.append(row)
        print(f"{name} R={R}: learn {learn_ms:.0f} ms | save {save_ms:.0f} ms, load {load_ms:.0f} ms, "
              f"read retained {read_ms:.0f} ms, request unlearn {req_ms:.0f} ms vs in-process {inproc_ms:.0f} ms "
              f"(merged equal: {same}, NaN rows {nan_rows}) | state {row['state_bytes'] / 2**20:.1f} MiB, checkpoints "
              f"{max(ck) / 2**20:.1f} MiB per shard", flush=True)
        del s, s2, L, data, tl
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--out', default=None)
    ap.add_argument('--skip-c3', action='store_true')
    ap.add_argument('--dir', default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.zeros(1, device='cuda')
    root = a.dir or tempfile.mkdtemp(prefix='prof_state_')
    res = dict(card=card())
    print('card:', res['card'], flush=True)
    try:
        res['ml1m'] = scenario('ml1m', *synth.ml_like(), 6040, 3416, 5, 16, 50, root)
        if not a.skip_c3:
            rng = np.random.default_rng(1)
            U, I = 138_493, 26_744
            mk = lambda n: (np.sort(rng.integers(0, U, n)), rng.integers(0, I, n), rng.integers(1, 6, n).astype(float))
            train, test = mk(20_000_000), mk(2_000_000)
            res['c3'] = scenario('c3', train, test, U, I, 8, 64, 50, root)
    finally:
        if a.dir is None:
            shutil.rmtree(root, ignore_errors=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
