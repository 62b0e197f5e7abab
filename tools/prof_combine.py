"""The learned combination of the SISA shard models on the GPU: times of the fit, the group scoring and the per-group
top-N, and the accuracy of three weightings on the ml1m-shaped synthetic set.

    python tools/prof_combine.py [--reps 10] [--epochs 50] [--json OUT]

Times (CUDA events, warmed up, mean over --reps), at the ml1m shape (6040 x 3416, K = 5, d = 16, 900 000 training and
100 000 test rows) and the C3 shape (138 493 x 26 744, K = 8, d = 64, 20 M training and 2 M test rows), random N(0, 1)
tables and uniform records, users spread over K owner groups:
  gram      ure_combine_gram over every group's training rows (one call)
  fit       utils.fit_combination: the Gram, its read-back, the host solve and ure_item_wsum of the K + 1 tables
  score     ure_group_score of the test rows
  topn      per owner group ure_topn on T_g plus b_g (what utils.recommend_combined runs): N = 10 for every user,
            seen lists = the training rows, built once outside the window
Accuracy: Sisa.learn on synth.ml_like with K = 5 uniform groups and --epochs epochs, then test RMSE / NDCG@10 / HR@10
and full-catalogue top-10 HR / Recall / NDCG for the mean (1/K sum_k), the fitted combination, and owner-only (one-hot
w, b = 0, through the same ure_group_score and per-group top-N).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ultrare_b200 import kernels as kn  # noqa: E402
from ultrare_b200.method import utils as ut  # noqa: E402

SHAPES = {   # name: (n_user, n_item, K, d, training rows, test rows)
    "ml1m": (6040, 3416, 5, 16, 900_000, 100_000),
    "c3": (138493, 26744, 8, 64, 20_000_000, 2_000_000),
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in q.split(",")]
    return name, float(power)


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps, out


def _records(g, n_user, n_item, n, users_of, dev):
    rec = torch.zeros((n, 4), dtype=torch.int32, device=dev)
    rec[:, 0] = users_of[torch.randint(0, users_of.shape[0], (n,), generator=g, device=dev)]
    rec[:, 1] = torch.randint(0, n_item, (n,), generator=g, device=dev, dtype=torch.int32)
    rec[:, 2] = (torch.randint(1, 6, (n,), generator=g, device=dev).float() / 5).view(torch.int32)
    return rec


def run_shape(name, reps):
    n_user, n_item, K, d, n_train, n_test = SHAPES[name]
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(0)
    P = torch.randn((n_user, d), generator=g, device=dev)
    Qs = [torch.randn((n_item, d), generator=g, device=dev) for _ in range(K)]
    owner = (torch.arange(n_user, device=dev, dtype=torch.int32) % K).contiguous()
    recs = [_records(g, n_user, n_item, n_train // K, torch.nonzero(owner == k).flatten().int(), dev) for k in range(K)]
    test = _records(g, n_user, n_item, n_test, torch.arange(n_user, device=dev, dtype=torch.int32), dev)
    gram_ms, _ = timed(lambda: kn.combine_gram(P, Qs, recs), reps)
    fit_ms, comb = timed(lambda: ut.fit_combination(P, Qs, recs), reps)
    score_ms, _ = timed(lambda: kn.group_score(P, comb.T, comb.b_slot, owner, test), reps)
    seen = kn.seen_lists(recs, n_user, n_item)                  # built once, outside the timed window
    slot = owner.long()
    groups = [torch.nonzero(slot == k).flatten().int() for k in range(K)]

    def topn():        # what utils.recommend_combined runs per owner group: ure_topn on T_g, then + b_g
        out = []
        for k, ug in enumerate(groups):
            items, sc = kn.recommend_topn(P, comb.T[k], ug, 10, 1.0, seen)
            out.append(torch.where(items >= 0, sc + comb.b_slot[k], sc))
        return out
    topn_ms, _ = timed(topn, max(1, reps // 2))
    return dict(shape=name, n_user=n_user, n_item=n_item, K=K, d=d, train_rows=n_train, test_rows=n_test,
                gram_ms=gram_ms, fit_ms=fit_ms, score_ms=score_ms, topn_ms=topn_ms)


def accuracy(epochs):
    """mean / fit / owner-only on ml1m-shaped synthetic data after `epochs` epochs of SISA training."""
    import pandas as pd
    from ultrare_b200 import synth
    from ultrare_b200.method.sisa import Sisa
    from ultrare_b200.read import RatingData, loadData, readRating
    U, I, K, B = 6040, 3416, 5, 30000
    train, test = synth.ml_like()
    trr, groups = readRating(pd.DataFrame({0: train[0], 1: train[1], 2: train[2]}), U, 5, [], [], K, [], 'a')
    ter, _ = readRating(pd.DataFrame({0: test[0], 1: test[1], 2: test[2]}), U, 5, [], [], K, groups)

    class Param:
        n_user, n_item, k, lam, seed, lr, lr_decay, momentum, batch = U, I, 16, 0.1, 42, 0.001, 0.95, 0.9, B
    Param.epochs = epochs
    tl = [loadData(RatingData(a), B, 1, True) for a in trr]
    sl = [loadData(RatingData(a), B, 1, False) for a in ter]
    total = loadData(RatingData(np.hstack(ter)), B, 1, False)
    s = Sisa(Param, 'mf', K, groups)
    s.epoch_eval = 'none'
    s.combine = 'fit'
    s.learn(tl, sl, total, 0, '')
    dev = s.device
    P = s.model_list[0].user_mat.weight.data
    Qs = [m.item_mat.weight.data for m in s.model_list]
    fit = s.combination
    one_hot = np.concatenate([np.eye(K), np.full((1, K), 1.0 / K)]).astype(np.float32)
    owner_only = ut.Combination(np.eye(K), np.zeros(K), kn.item_wsum(Qs, kn.upload_array(one_hot, dev)),
                                torch.zeros(K + 1, dtype=torch.float32, device=dev), None)
    out = {"fit_w": fit.w.tolist(), "fit_b": fit.b.tolist()}
    s.combine = 'mean'
    rmse, ndcg, hr = s._ensemble_test(total, 0)
    items, _ = s.recommend(None, 10, exclude=tl)
    out["mean"] = dict(rmse=rmse, ndcg=ndcg, hr=hr, top10=ut.topn_metrics(items, None, total, 10))
    s.combine = 'fit'
    for name, c in (("fit", fit), ("owner", owner_only)):
        s.combination = c
        rmse, ndcg, hr = s._combined_test(total, 0)
        items, _ = s.recommend(None, 10, exclude=tl)
        out[name] = dict(rmse=rmse, ndcg=ndcg, hr=hr, top10=ut.topn_metrics(items, None, total, 10))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--epochs", type=int, default=50)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_combine: needs a CUDA device")
    name, power = card()
    rows = [run_shape(s, a.reps) for s in SHAPES]
    hdr = ("shape", "K", "d", "train_rows", "gram_ms", "fit_ms", "score_ms", "topn_ms")
    print(" | ".join(hdr))
    for r in rows:
        print(" | ".join(f"{r[k]:.4g}" if isinstance(r[k], float) else str(r[k]) for k in hdr))
    acc = accuracy(a.epochs)
    print(f"ml1m synthetic, K = 5, {a.epochs} epochs:")
    for w in ("mean", "fit", "owner"):
        m = acc[w]
        t = m["top10"]
        print(f"  {w:6s} test RMSE {m['rmse']:.4f} NDCG@10 {m['ndcg']:.4f} HR@10 {m['hr']:.4f} | top-10 HR {t['hr']:.4f} "
              f"Recall {t['recall']:.4f} NDCG {t['ndcg']:.4f}")
    print("  fit w:", np.round(np.asarray(acc["fit_w"]), 4).tolist(), "b:", np.round(np.asarray(acc["fit_b"]), 4).tolist())
    print(f"card: {name}, power limit {power:.0f} W")
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            json.dump(dict(card=name, power_limit_w=power, times=rows, accuracy=acc, epochs=a.epochs), f, indent=1)


if __name__ == "__main__":
    main()
