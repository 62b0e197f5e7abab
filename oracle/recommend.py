"""Float64 NumPy restatement of top-N recommendation over the whole catalogue and its metrics (test-only; the
product never imports it).

score(u, i) = scale * sum_t P[u,t] * S[i,t]; a user's seen items are never returned; order: score descending, ties
to the smaller item id; lists shorter than N are padded with item -1 / score -inf.  Metrics: relevant items are a
user's distinct test items with normalised rating >= 4/5 (reference utils.py:175,180); users without one are not
counted; HR@N = any hit, Recall@N = hits / |rel|, NDCG@N = sum_{p<N, hit} 1/log2(p+2) / sum_{p<min(N,|rel|)} 1/log2(p+2).
"""
from __future__ import annotations

import numpy as np


def scores(P, S, users, scale):
    """float64 [m, n_item] scores of the requested users."""
    return scale * (np.asarray(P, np.float64)[np.asarray(users)] @ np.asarray(S, np.float64).T)


def seen_sets(records, n_user):
    """list of per-user sets of item ids from (user, item, ...) records."""
    out = [set() for _ in range(n_user)]
    for u, i in np.asarray(records)[:, :2]:
        out[int(u)].add(int(i))
    return out


def topn(P, S, users, top_n, scale, seen=None):
    """(items int64 [m, N], scores float64 [m, N], eligible count [m]) of the oracle."""
    sc = scores(P, S, users, scale)
    m, n_item = sc.shape
    items = np.full((m, top_n), -1, dtype=np.int64)
    vals = np.full((m, top_n), -np.inf)
    n_ok = np.zeros(m, dtype=np.int64)
    for r, u in enumerate(np.asarray(users)):
        ok = np.ones(n_item, dtype=bool)
        if seen is not None and seen[int(u)]:
            ok[list(seen[int(u)])] = False
        cand = np.flatnonzero(ok)
        order = cand[np.lexsort((cand, -sc[r, cand]))]        # score descending, then item ascending
        k = min(top_n, len(order))
        items[r, :k] = order[:k]
        vals[r, :k] = sc[r, order[:k]]
        n_ok[r] = len(cand)
    return items, vals, n_ok


def metrics(items, users, test_records, top_n):
    """dict(hr, recall, ndcg, users): sums over counted users (not averages)."""
    rel = {}
    for u, i, r in ((int(a), int(b), float(c)) for a, b, c in
                    zip(test_records[:, 0], test_records[:, 1], test_records[:, 2])):
        if r >= 4.0 / 5.0:
            rel.setdefault(u, set()).add(i)
    w = 1.0 / np.log2(np.arange(2, top_n + 2))
    hr = recall = ndcg = cnt = 0.0
    for row, u in enumerate(np.asarray(users)):
        R = rel.get(int(u))
        if not R:
            continue
        lst = [int(x) for x in items[row, :top_n]]
        hit = np.array([x >= 0 and x in R for x in lst], dtype=bool)
        hr += float(hit.any())
        recall += hit.sum() / len(R)
        ndcg += w[hit].sum() / w[:min(top_n, len(R))].sum()
        cnt += 1
    return dict(hr=hr, recall=recall, ndcg=ndcg, users=cnt)
