"""ure_rank_metrics alone at the ml1m test shape: device time of one call (HR@10 / NDCG@10 over every user's rows).

    python tools/prof_eval.py [--reps 200] [--json OUT]

Test set: the ~10 % per-user test split of synth.ml_like (6 040 users, ~100 k rows), N(0,1) fp32 scores.  Three cases:
rows in user order (identity segments); rows shuffled and ranked through the order of ure_user_segments (what the
SISA evaluation passes); the shuffled rows with the scores of 1 088 users NaN (the merged table a diverged sliced
unlearn leaves at ml1m).  Time: CUDA events around --reps back-to-back calls after a warm-up, mean per call.  The
card's name and power limit are read in the same run.
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
from ultrare_b200 import kernels as kn, synth  # noqa: E402


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
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    _, (u, _, r) = synth.ml_like()
    n, n_user = len(u), int(u.max()) + 1
    rng = np.random.default_rng(0)
    s = rng.standard_normal(n).astype(np.float32)
    r32 = (r / 5.0).astype(np.float32)
    out = torch.zeros(3, dtype=torch.float64, device=dev)
    res = {"n_rows": n, "n_users": n_user, "reps": args.reps}
    inter = kn.pack_interactions(u, np.zeros(n, dtype=np.int64), r32, dev)
    seg = kn.upload_array(np.concatenate([[0], np.cumsum(np.bincount(u, minlength=n_user))]).astype(np.int64), dev)
    score = torch.tensor(s, device=dev)
    res["user_order_us"] = 1e3 * timed(lambda: kn.rank_metrics(inter, score, seg, out=out), args.reps)
    p = rng.permutation(n)
    inter = kn.pack_interactions(u[p], np.zeros(n, dtype=np.int64), r32[p], dev)
    order, seg = kn.user_segments_device(inter, n_user)
    score = torch.tensor(s[p], device=dev)
    res["shuffled_us"] = 1e3 * timed(lambda: kn.rank_metrics(inter, score, seg, order, out=out), args.reps)
    nan_users = rng.choice(n_user, 1088, replace=False)
    score = torch.tensor(np.where(np.isin(u[p], nan_users), np.float32(np.nan), s[p]), device=dev)
    res["shuffled_nan_users_us"] = 1e3 * timed(lambda: kn.rank_metrics(inter, score, seg, order, out=out),
                                              args.reps)
    res["card"], res["power_limit_w"] = card()
    line = json.dumps(res)
    print(line)
    if args.json:
        with open(args.json, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
