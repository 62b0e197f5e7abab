"""What BPR training (loss='bpr', ure_mf_train_bpr) costs and what it gives on catalogue top-10.

    python tools/prof_bpr.py [--out result.json] [--epochs 50] [--skip-c3] [--skip-accuracy]

Step throughput, CUDA events around E_t epochs after one warm-up epoch, for three schedules on the same shards:
MSE DENSE, MSE auto (OWNER where it fits) and BPR (DENSE).  Shapes (users split by id mod K, compact user tables):
  * ml1m: 6040 users x 3416 items, 900 k rows, K = 5, d = 16, batch 30 000;
  * C3 share: 138 493 users x 26 744 items, 20 M rows (synth.device_interactions), K = 8, d = 64, batch 30 000.
Rates are triples (interactions) per second; the share of the copy peak credits 16 + 24 d bytes per triple (the
record, three gathered rows and three scattered rows, fp32) against 7.7 TB/s.
Sampler cost: candidates drawn per triple and dropped triples (ure_bpr_negatives, epoch 0) on synth.ml_like, K = 5.
Accuracy: full-catalogue top-10 HR / Recall / NDCG on synth.ml_like (rec10_metrics.npy of main.py --recommend 10) for
MSE and BPR, Scratch (--group 0) and Sisa K = 5 with the mean (rating-ot grouping, learn pass), --epoch E.
The card name and power limit are printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ultrare_b200 import kernels as kn, synth                                 # noqa: E402


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ''
    return q or torch.cuda.get_device_name(0) + ', power limit unknown'


def split(rec, K):
    """Records by user id mod K, user field -> row u // K of the shard's table."""
    out = []
    for s in range(K):
        r = rec[rec[:, 0] % K == s].clone()
        r[:, 0] //= K
        out.append(r.contiguous())
    return out


def throughput(rec, n_user, n_item, K, d, epochs_timed, dev):
    recs = split(rec, K)
    rows = [-(-n_user // K)] * K
    res = {}
    for name, mode, loss in (("mse_dense", "dense", "mse"), ("mse_auto", "auto", "mse"), ("bpr", "dense", "bpr")):
        sb = kn.ArenaShardBatch(recs, rows, n_item, d, 30000, 1 + epochs_timed, list(range(1, K + 1)), 42,
                                mode=mode, std=0.1, loss=loss)
        spe = sb.total_steps // (1 + epochs_timed)
        sb.train(spe)                                             # warm-up epoch
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        sb.train()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        triples = sum(int(r.shape[0]) for r in recs) * epochs_timed
        res[name] = dict(schedule=sb.mode, ms=round(ms, 3), steps=sb.total_steps - spe,
                         triples_per_s=triples / (ms / 1e3),
                         copy_peak_share=triples * (16 + 24 * d) / (ms / 1e3) / 7.7e12)
        del sb
    return res


def sampler(rec, n_item, K):
    tries, dropped, n = 0, 0, 0
    for s, r in enumerate(split(rec, K)):
        seen = kn.seen_lists(r, int(r[:, 0].max()) + 1, n_item)
        neg, t = kn.bpr_negatives(r, n_item, seen, 42, s + 1, 0, want_tries=True)
        tries += int(t.sum())
        dropped += int((neg < 0).sum())
        n += int(r.shape[0])
    return dict(mean_candidates=tries / n, dropped=dropped, triples=n)


def accuracy(epochs):
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        env = dict(os.environ, ULTRARE_ROOT=tmp)
        for loss in ("mse", "bpr"):
            for group in (0, 5):
                args = [sys.executable, os.path.join(ROOT, "main.py"), "--dataset", "ml1m", "--synth", "--group",
                        str(group), "--epoch", str(epochs), "--verbose", "0", "--recommend", "10", "--loss", loss]
                if group:
                    args += ["--grouping", "rating-ot", "--epoch-eval", "none"]
                r = subprocess.run(args, cwd=ROOT, env=env, capture_output=True, text=True)
                if r.returncode != 0:
                    raise RuntimeError(r.stdout[-2000:] + r.stderr[-4000:])
                run = "ml1m_g%d%s" % (group, "_bpr" if loss == "bpr" else "")
                sub = "MF_full_train" if group == 0 else "MF_rating-ot_sisa_learn"
                m = np.load(os.path.join(tmp, "result", "2", "rand", run, sub, "rec10_metrics.npy"))
                out[f"{loss}_{'scratch' if group == 0 else 'sisa5_mean'}"] = dict(hr=m[0], recall=m[1], ndcg=m[2])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--epochs", type=int, default=50)
    ap.add_argument("--skip-c3", action="store_true")
    ap.add_argument("--skip-accuracy", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_bpr.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    res = {"card": card()}
    tr, _ = synth.ml_like()
    ml = kn.pack_interactions(tr[0], tr[1], tr[2] / 5.0, dev)
    res["ml1m"] = throughput(ml, 6040, 3416, 5, 16, 10, dev)
    res["sampler_ml1m"] = sampler(ml, 3416, 5)
    print(json.dumps(res, indent=1), flush=True)
    if not a.skip_c3:
        c3 = synth.device_interactions(138493, 26744, 20_000_000, dev)
        res["c3"] = throughput(c3, 138493, 26744, 8, 64, 3, dev)
        res["sampler_c3"] = sampler(c3, 26744, 8)
        del c3
        print(json.dumps({k: res[k] for k in ("c3", "sampler_c3")}, indent=1), flush=True)
    if not a.skip_accuracy:
        res["top10_synth_ml_like"] = accuracy(a.epochs)
    res["card_after"] = card()
    text = json.dumps(res, indent=1, default=float)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
