"""Float64 NumPy restatement of the learned combination of the SISA shard models (test-only; the product never
imports it).

Owner group g = the users whose owner shard is g.  For a rating (u, i, r): x_k = P[u].Q_k[i], k < K, P the merged user
table.  Score s(u, i) = b_g + sum_k w_gk x_k = b_g + P[u].T_g[i], T_g = sum_k w_gk Q_k.  Fit of group g on its
training rows: min sum (b_g + w_g.x - r)^2 + lambda_g ||w_g||^2, lambda_g = 1e-6 tr(X_g^T X_g) / K, the intercept not
penalised, solved from the (K+1) x (K+1) normal equations.  A group without rows, and a user in no group, use the
mean combination w = 1/K, b = 0.
"""
from __future__ import annotations

import numpy as np

from . import recommend as orec

RIDGE = 1e-6


def features(P, Qs, users, items):
    """float64 [n, K]: x_k = P[u].Q_k[i] from the (fp32) tables."""
    P = np.asarray(P, np.float64)[np.asarray(users, np.int64)]
    return np.stack([(P * np.asarray(Q, np.float64)[np.asarray(items, np.int64)]).sum(1) for Q in Qs], 1) \
        if len(users) else np.zeros((0, len(Qs)))


def gram(X, r):
    """(G = sum [x;1][x;1]^T  [(K+1), (K+1)], m = sum [x;1] r  [K+1], n)."""
    Z = np.concatenate([X, np.ones((X.shape[0], 1))], 1)
    r = np.asarray(r, np.float64)
    return Z.T @ Z, Z.T @ r, X.shape[0]


def solve(G, m, n, K):
    """(w [K], b) of the ridge fit from the normal equations; the mean for a group without rows."""
    if n == 0:
        return np.full(K, 1.0 / K), 0.0
    A = np.array(G, np.float64)
    A[np.arange(K), np.arange(K)] += RIDGE * np.trace(A[:K, :K]) / K
    th = np.linalg.solve(A, m)
    return th[:K], th[K]


def fit(P, Qs, group_rows):
    """(w [K, K], b [K]): group_rows[g] = (users, items, ratings) of group g's training rows."""
    K = len(Qs)
    w, b = np.zeros((K, K)), np.zeros(K)
    for g, (u, i, r) in enumerate(group_rows):
        w[g], b[g] = solve(*gram(features(P, Qs, u, i), r), K)
    return w, b


def _weights(w, b, owner, users):
    """Per-row (w, b) of the users' groups; the mean for users in no group."""
    K = w.shape[1]
    g = np.asarray(owner)[np.asarray(users, np.int64)]
    W = np.where((g >= 0)[:, None], w[np.maximum(g, 0)], 1.0 / K)
    return W, np.where(g >= 0, b[np.maximum(g, 0)], 0.0)


def scores(P, Qs, w, b, owner, users, items):
    """float64 [n] combined scores of (users, items)."""
    W, B = _weights(w, b, owner, users)
    return B + (features(P, Qs, users, items) * W).sum(1)


def item_tables(Qs, w):
    """float64 [G, n_item, d]: T_g = sum_k w[g, k] Q_k for every row g of w."""
    Q = np.stack([np.asarray(q, np.float64) for q in Qs])
    return np.einsum('gk,kid->gid', np.asarray(w, np.float64), Q)


def topn(P, Qs, w, b, owner, users, top_n, seen=None):
    """(items [m, N], scores [m, N]) per requested user: oracle.recommend.topn of the user's group (T_g, scale 1) plus
    b_g, -1 / -inf padding unchanged; users in no group with the mean combination."""
    K = len(Qs)
    users = np.asarray(users, np.int64)
    g = np.asarray(owner)[users]
    slot = np.where(g >= 0, g, K)
    T = item_tables(Qs, np.concatenate([w, np.full((1, K), 1.0 / K)]))
    B = np.append(b, 0.0)
    items = np.full((len(users), top_n), -1, dtype=np.int64)
    vals = np.full((len(users), top_n), -np.inf)
    for s in np.unique(slot):
        rows = np.flatnonzero(slot == s)
        it, sc, _ = orec.topn(P, T[s], users[rows], top_n, 1.0, seen)
        items[rows] = it
        vals[rows] = np.where(it >= 0, sc + B[s], sc)
    return items, vals
