"""Oracle: BPR training of one shard model (ure_mf_train_bpr), restated in NumPy fp32.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

For record idx = (user row u, item i) of the records the launch trains, in epoch e:
  * sampler (ultrare_b200/csrc/bpr_sampler.cuh), uint32 arithmetic:
        key = perm_key(perm_seed, shard_id, e)                       (oracle/mf.py)
        h   = mix32(key ^ (idx * 0x9E3779B1 + 0x7F4A7C15))
        c_t = mulhi32(mix32(h + t * 0x85EBCA77), n_item)             t = 0 .. 15
    the negative j is the first c_t not among u's items in those records; none: the triple is dropped (j = -1);
  * x = P[u].(Q[i] - Q[j]); loss softplus(-x); with c = sigmoid(-x) the gradients -c (Q[i] - Q[j]) of P[u],
    -c P[u] of Q[i] and +c P[u] of Q[j], all from the pre-step weights, summed over the batch;
  * then the unchanged dense SGD (momentum, L2) of oracle/mf.py's sgd_dense and StepLR, on every batch of the
    visiting order (a batch whose triples are all dropped still takes its weight-decay / momentum step);
  * the epoch's train loss is the summed softplus(-x) / n, dropped triples counting zero.
"""
from __future__ import annotations

import numpy as np

from .mf import lr_at_epoch, mix32, perm_key, sgd_dense

CANDIDATES = 16
_M = 0xFFFFFFFF


def record_hash(key: int, idx) -> np.ndarray:
    idx = np.asarray(idx, dtype=np.uint64)
    return mix32(np.uint64(key) ^ ((idx * 0x9E3779B1 + 0x7F4A7C15) & _M))


def candidates(key: int, n: int, n_item: int) -> np.ndarray:
    """uint64 [n, CANDIDATES]: the candidates c_t of records 0 .. n-1."""
    h = record_hash(key, np.arange(n))[:, None]
    t = np.arange(CANDIDATES, dtype=np.uint64)[None, :]
    return (mix32((h + t * 0x85EBCA77) & _M) * np.uint64(n_item)) >> 32


def negatives(u, i, n_item: int, perm_seed: int, shard_id: int, epoch: int, return_tries: bool = False):
    """int64 [n]: the negative of every record (-1: dropped), the seen lists being the items of (u, i) themselves."""
    u = np.asarray(u, dtype=np.int64)
    i = np.asarray(i, dtype=np.int64)
    n = len(u)
    c = candidates(perm_key(perm_seed, shard_id, epoch), n, n_item).astype(np.int64)
    seen = np.unique(u * n_item + i)
    key = u[:, None] * n_item + c
    pos = np.searchsorted(seen, key)
    hit = (pos < len(seen)) & (seen[np.minimum(pos, len(seen) - 1)] == key) if len(seen) else np.zeros_like(key, bool)
    free = ~hit
    first = np.argmax(free, axis=1)
    ok = free[np.arange(n), first] if n else np.zeros(0, bool)
    neg = np.where(ok, c[np.arange(n), first], -1)
    if return_tries:
        return neg, np.where(ok, first + 1, CANDIDATES)
    return neg


def softplus(x):
    return np.logaddexp(np.float32(0), -x).astype(np.float32)


def bpr_train_epoch(P, Q, bufP, bufQ, u, i, neg, perm, batch, lr, wd, mu, step0):
    """One BPR epoch in place; returns the summed softplus(-x) of the epoch's triples."""
    f = np.float32
    total = 0.0
    step = step0
    n = len(u)
    for s in range(0, n, batch):
        idx = perm[s:s + batch]
        idx = idx[neg[idx] >= 0]
        ub, ib, jb = u[idx], i[idx], neg[idx]
        pu, qd = P[ub], Q[ib] - Q[jb]
        x = (pu * qd).sum(axis=1, dtype=f)
        total += float(softplus(x).sum(dtype=np.float64))
        c = (f(1) / (f(1) + np.exp(x))).astype(f)[:, None]
        gP = np.zeros_like(P)
        gQ = np.zeros_like(Q)
        np.add.at(gP, ub, -c * qd)
        np.add.at(gQ, ib, -c * pu)
        np.add.at(gQ, jb, c * pu)
        sgd_dense(P, bufP, gP, lr, wd, mu, step == 0)
        sgd_dense(Q, bufQ, gQ, lr, wd, mu, step == 0)
        step += 1
    return total


def bpr_train(P0, Q0, u, i, perms, batch, epochs, perm_seed, shard_id, lr0=1e-3, wd=0.1, mu=0.9, lr_decay=0.95):
    """BPR training of one shard: (P, Q, bufP, bufQ, losses) with losses[e] = summed softplus(-x) / n."""
    P, Q = P0.astype(np.float32).copy(), Q0.astype(np.float32).copy()
    bufP, bufQ = np.zeros_like(P), np.zeros_like(Q)
    u = np.asarray(u, dtype=np.int64)
    i = np.asarray(i, dtype=np.int64)
    n = len(u)
    losses, step = [], 0
    for ep in range(epochs):
        neg = negatives(u, i, Q.shape[0], perm_seed, shard_id, ep)
        tot = bpr_train_epoch(P, Q, bufP, bufQ, u, i, neg, perms[ep], batch, lr_at_epoch(lr0, lr_decay, ep), wd, mu,
                              step)
        step += -(-n // batch)
        losses.append(tot / max(1, n))
    return P, Q, bufP, bufQ, np.asarray(losses)
