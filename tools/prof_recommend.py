"""Top-N recommendation (ure_topn) on the GPU: kernel time, scores/s, the bound, and a chunked fp32 torch baseline.

    python tools/prof_recommend.py [--reps 20] [--only ml1m,c3,...] [--json OUT]

Shapes: ml1m (6040 x 3416, d = 16, N = 10), C3 (138 493 x 26 744, d = 64, N = 10 and 50), a large catalogue
(200 000 users x 10^6 items, d = 128, N = 10) and single-user latency over 10^6 items.  Random N(0,1) tables, about
20 seen items per user.  Kernel time: CUDA events around split-lo + top-N (+ merge), warmed up, mean over --reps.
Bound: the largest of the tensor time (6 d flops per score -- three tf32 products of 2 d flops -- against the
data-sheet 1,125 TFLOP/s dense TF32, a data-sheet figure, not a measured one), the epilogue issue time (~1.25
instructions per score -- tcgen05.ld share, one max, one compare -- on 4 x 32 lanes per SM per clock at the card's
maximum SM clock) and the HBM time (S read, S_lo written and read, user rows, lists: against the data-sheet
7.7 TB/s).  Baseline: P[users] @ S.T in fp32 (TF32 off) in chunks, seen items masked to -inf, torch.topk; its lists
are compared with the kernel's.
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

SHAPES = {   # name: (n_user requested, n_user table, n_item, d, N)
    "ml1m": (6040, 6040, 3416, 16, 10),
    "c3_n10": (138493, 138493, 26744, 64, 10),
    "c3_n50": (138493, 138493, 26744, 64, 50),
    "large": (200000, 200000, 1000000, 128, 10),
    "one_user": (1, 200000, 1000000, 128, 10),
}
TF32_PEAK = 1125e12
HBM_PEAK = 7.7e12
EPI_INSTR_PER_SCORE = 1.25


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clk = [x.strip() for x in q.split(",")]
    return name, float(power), float(clk)


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


def baseline(P, S, users, N, scale, seen_mask_rows, chunk_bytes=2 << 30):
    torch.backends.cuda.matmul.allow_tf32 = False
    m, n_item = users.shape[0], S.shape[0]
    rows = max(1, min(m, chunk_bytes // (4 * n_item)))
    items = torch.empty((m, N), dtype=torch.int64, device=P.device)
    scores = torch.empty((m, N), dtype=torch.float32, device=P.device)
    for r0 in range(0, m, rows):
        r1 = min(m, r0 + rows)
        sc = (P[users[r0:r1].long()] @ S.T) * scale
        seen_mask_rows(sc, r0, r1)
        k = min(N, n_item)
        v, i = torch.topk(sc, k, dim=1)
        items[r0:r1, :k], scores[r0:r1, :k] = i, v
    return items, scores


def run(name, reps):
    m, n_user, n_item, d, N = SHAPES[name]
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(0)
    P = torch.randn((n_user, d), generator=g, device=dev)
    S = torch.randn((n_item, d), generator=g, device=dev)
    users = torch.arange(m, dtype=torch.int32, device=dev) if m == n_user else \
        torch.randint(0, n_user, (m,), generator=g, device=dev, dtype=torch.int32)
    n_rec = 20 * n_user
    rec = torch.zeros((n_rec, 4), dtype=torch.int32, device=dev)
    rec[:, 0] = torch.randint(0, n_user, (n_rec,), generator=g, device=dev, dtype=torch.int32)
    rec[:, 1] = torch.randint(0, n_item, (n_rec,), generator=g, device=dev, dtype=torch.int32)
    seen = kn.seen_lists(rec, n_user, n_item)
    scale = 0.2
    ms, (items, scores) = timed(lambda: kn.recommend_topn(P, S, users, N, scale, seen), reps)
    torch.cuda.synchronize()
    off, sitems = seen

    def mask(sc, r0, r1):
        u = users[r0:r1].long()
        lo, hi = off[u], off[u + 1]
        cnt = hi - lo
        rows = torch.repeat_interleave(torch.arange(r1 - r0, device=dev), cnt)
        pos = torch.arange(int(cnt.sum()), device=dev) - torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
        sc[rows, sitems[torch.repeat_interleave(lo, cnt) + pos].long()] = -float("inf")

    bms, (bi, bs) = timed(lambda: baseline(P, S, users, N, scale, mask), 1 if n_item * m > 1e10 else max(1, reps // 4))
    same_lists = float((bi == items.long()).all(1).float().mean())
    max_score_diff = float((bs - scores).abs().max())
    n_scores = m * n_item
    name_, power, clk = card()
    t_tensor = 6 * d * n_scores / TF32_PEAK
    t_epi = EPI_INSTR_PER_SCORE * n_scores / (torch.cuda.get_device_properties(0).multi_processor_count * 128 * clk * 1e6)
    t_hbm = (3 * n_item * d * 4 + m * d * 4 + m * N * 8) / HBM_PEAK
    bounds = {"tensor": t_tensor, "epilogue": t_epi, "hbm": t_hbm}
    bound = max(bounds, key=bounds.get)
    return dict(shape=name, m=m, n_item=n_item, d=d, N=N, kernel_ms=ms, scores_per_s=n_scores / (ms * 1e-3),
                tensor_bound_ms=t_tensor * 1e3, epilogue_bound_ms=t_epi * 1e3, hbm_bound_ms=t_hbm * 1e3, bound=bound,
                share_of_bound=bounds[bound] * 1e3 / ms, torch_ms=bms, speedup=bms / ms,
                torch_same_lists=same_lists, torch_max_score_diff=max_score_diff,
                card=name_, power_limit_w=power, max_sm_clock_mhz=clk)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--only", default=",".join(SHAPES))
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_recommend: needs a CUDA device")
    rows = [run(s, a.reps) for s in a.only.split(",")]
    hdr = ("shape", "kernel_ms", "scores_per_s", "bound", "tensor_bound_ms", "epilogue_bound_ms", "hbm_bound_ms",
           "share_of_bound", "torch_ms", "speedup", "torch_same_lists")
    print(" | ".join(hdr))
    for r in rows:
        print(" | ".join(f"{r[k]:.4g}" if isinstance(r[k], float) else str(r[k]) for k in hdr))
    print(f"card: {rows[0]['card']}, power limit {rows[0]['power_limit_w']:.0f} W, max SM clock "
          f"{rows[0]['max_sm_clock_mhz']:.0f} MHz")
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
