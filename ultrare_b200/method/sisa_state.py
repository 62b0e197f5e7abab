"""The on-disk state of a trained SISA model and the ledger of the deletions applied to it (DESIGN.md §4.10).

A state directory holds ``.npy`` arrays (read with allow_pickle=False) and one ``manifest.json`` written last: its
presence marks the directory complete.  Sisa.save_state / Sisa.load_state / Sisa.apply_request use the helpers here;
everything in this module runs on the host.
"""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np

FORMAT_VERSION = 1
MANIFEST = 'manifest.json'
# manifest keys every state carries (load_state refuses a manifest without one of them)
MANIFEST_KEYS = ('format', 'K', 'slices', 'k', 'n_user', 'n_item', 'epochs', 'batch', 'lr', 'lr_decay', 'lam',
                 'momentum', 'seed', 'combine', 'epoch_eval', 'dataset', 'grouping', 'max_rating', 'train_file',
                 'test_file', 'requests')


def file_digest(path, chunk=1 << 24):
    """(size in bytes, sha256 hex) of a file."""
    h = hashlib.sha256()
    with open(path, 'rb') as f:
        while True:
            b = f.read(chunk)
            if not b:
                break
            h.update(b)
    return os.path.getsize(path), h.hexdigest()


def flat_index(groups):
    """A list of user-id lists as (ids int64 [n], offsets int64 [len + 1])."""
    lens = [len(g) for g in groups]
    ids = np.concatenate([np.asarray(g, dtype=np.int64) for g in groups]) if groups else np.zeros(0, dtype=np.int64)
    return ids.astype(np.int64), np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)


def unflat_index(ids, off):
    return [ids[int(off[g]):int(off[g + 1])].tolist() for g in range(len(off) - 1)]


def load_array(state_dir, name):
    path = os.path.join(state_dir, name + '.npy')
    if not os.path.exists(path):
        raise ValueError(f"{state_dir} is not a complete SISA state: {name}.npy is missing")
    return np.load(path, allow_pickle=False)


def read_manifest(state_dir):
    """The manifest of a complete state of this format; ValueError when the directory holds none, an incomplete one or
    one of another format version."""
    path = os.path.join(state_dir, MANIFEST)
    if not os.path.exists(path):
        raise ValueError(f"{state_dir} is not a complete SISA state: it has no {MANIFEST}")
    try:
        with open(path) as f:
            man = json.load(f)
    except (OSError, ValueError) as e:
        raise ValueError(f"{path} cannot be read as JSON: {e}") from None
    if not isinstance(man, dict):
        raise ValueError(f"{path} is not a SISA state manifest")
    if man.get('format') != FORMAT_VERSION:
        raise ValueError(f"{path} has format version {man.get('format')!r}; this build reads version {FORMAT_VERSION}")
    missing = [k for k in MANIFEST_KEYS if k not in man]
    if missing:
        raise ValueError(f"{path} is incomplete: it lacks {missing}")
    man.setdefault('loss', 'mse')           # the training objective; states written before BPR training were MSE
    if man['loss'] not in ('mse', 'bpr'):
        raise ValueError(f"{path} has loss {man['loss']!r}; this build trains 'mse' or 'bpr'")
    return man


def check_training_file(man):
    """ValueError unless the training file the manifest names is still there with the same size and sha256: the
    retained data of every later request is read from it."""
    tf = man['train_file']
    path = tf['path']
    if not os.path.exists(path):
        raise ValueError(f"the state's training file {path} does not exist")
    size, sha = file_digest(path)
    if size != tf['bytes'] or sha != tf['sha256']:
        raise ValueError(f"the training file {path} changed since the state was saved (sha256 {sha}, the state "
                         f"recorded {tf['sha256']})")


def check_train_index(got, want):
    """The reader's count-sorted grouping must be the one the state was trained with."""
    if len(got) != len(want) or any(list(map(int, a)) != list(map(int, b)) for a, b in zip(got, want)):
        raise ValueError("the training file's count-sorted grouping differs from the state's train_index: the "
                         "training file changed since the state was saved")


# ------------------------------------------------------------------------------------------------ requests
def parse_request_file(path, kind):
    """A request file as int64: kind 'users' -> [n] (one id per line), 'ratings' -> [n, 2] (``user,item`` per line).
    ``.npy`` files are read with allow_pickle=False; anything else as text, comma- or whitespace-separated."""
    if kind not in ('users', 'ratings'):
        raise ValueError(f"kind must be 'users' or 'ratings', not {kind!r}")
    if path.endswith('.npy'):
        a = np.load(path, allow_pickle=False)
    else:
        with open(path) as f:
            rows = [ln.replace(',', ' ').split() for ln in f if ln.strip() and not ln.lstrip().startswith('#')]
        a = np.array([[float(x) for x in r] for r in rows], dtype=np.float64) if rows else \
            np.zeros((0, 1 if kind == 'users' else 2))
        if kind == 'users':
            if a.ndim != 2 or a.shape[1] != 1:
                raise ValueError(f"{path}: a user file holds one id per line")
            a = a[:, 0]
    a = np.asarray(a)
    if a.size and not np.array_equal(a, np.round(a)):
        raise ValueError(f"{path}: ids must be integers")
    return (a.reshape(-1) if kind == 'users' else a).astype(np.int64)


def validate_request(users, pairs, n_user, n_item):
    """(users int64 [n] sorted unique, pairs int64 [n, 2] sorted unique) of a deletion request; ValueError for a
    negative id, a user outside [0, n_user), an item outside [0, n_item) or a pair array that is not [n, 2]."""
    u = np.asarray([] if users is None else users).reshape(-1)
    if u.size and not np.array_equal(u, np.round(u)):
        raise ValueError("deleted users must be integer ids")
    u = u.astype(np.int64)
    p = np.asarray(pairs if pairs is not None else [])
    if p.size == 0:
        p = np.zeros((0, 2), dtype=np.int64)
    if p.ndim != 2 or p.shape[1] != 2:
        raise ValueError(f"deleted ratings must be an int array [n, 2] of (user, item), got shape {p.shape}")
    if not np.array_equal(p, np.round(p)):
        raise ValueError("deleted ratings must hold integer ids")
    p = p.astype(np.int64)
    if (u < 0).any() or (p < 0).any():
        raise ValueError("deletion request: user and item ids must be non-negative")
    if (u >= n_user).any() or (p[:, 0] >= n_user).any():
        raise ValueError(f"deletion request: user ids must be below n_user = {n_user}")
    if (p[:, 1] >= n_item).any():
        raise ValueError(f"deletion request: item ids must be below n_item = {n_item}")
    return np.unique(u), np.unique(p, axis=0).reshape(-1, 2)


def effective_request(users, pairs, led_users, led_pairs):
    """The part of a validated request the ledger does not hold: users not deleted yet, pairs neither deleted yet nor
    belonging to a deleted user."""
    users = users[~np.isin(users, led_users)]
    keep = ~np.isin(pairs[:, 0], led_users)
    if len(led_pairs):
        keep &= ~np.isin(pair_keys(pairs), pair_keys(led_pairs))
    return users, pairs[keep]


def pair_keys(pairs):
    return (pairs[:, 0].astype(np.int64) << 32) | pairs[:, 1].astype(np.int64)


def ledger_union(led_users, led_pairs, users, pairs):
    """The ledger after a request: sorted unique users, sorted unique pairs."""
    return (np.union1d(led_users, users).astype(np.int64),
            np.unique(np.concatenate([led_pairs, pairs]).astype(np.int64), axis=0).reshape(-1, 2))


def deletion_table(users, pairs):
    """One int64 [n, 2] array of a request: (user, -1) per deleted user, then (user, item) per deleted rating."""
    return np.concatenate([np.stack([users, np.full(len(users), -1, dtype=np.int64)], 1).reshape(-1, 2),
                           pairs.reshape(-1, 2)]).astype(np.int64)


# ------------------------------------------------------------------------------------------------ retained data
def read_retained(source, n_user, n_group, n_slice, batch, del_users, del_pairs, device=None):
    """(train loaders, test loaders, test loader, train_index) of the state's training file minus the given
    deletions, read as Instance reads an unlearn pass: the device ingest, or the host split under URE_HOST_INGEST=1 or
    without a device; the test file with the resulting train_index."""
    import torch

    from ..read import RatingData, loadData, readRating, readRatingDevice
    gi, mr = source['group_index'], source['max_rating']
    du, dr = np.asarray(del_users, dtype=np.int64), np.asarray(del_pairs, dtype=np.int64).reshape(-1, 2)
    if os.environ.get('URE_HOST_INGEST', '0') == '1' or not torch.cuda.is_available():
        train, train_index = readRating(source['train_file'], n_user, mr, du, dr, n_group, gi, 'a', n_slice)
        test, _ = readRating(source['test_file'], n_user, mr, [], [], n_group, train_index)
        train, test, total = [RatingData(r) for r in train], [RatingData(r) for r in test], RatingData(np.hstack(test))
    else:
        dev = device if device is not None else 'cuda'
        train, train_index, _ = readRatingDevice(source['train_file'], n_user, mr, du, dr, n_group, gi, 'a', dev,
                                                 n_slice=n_slice)
        test, _, total = readRatingDevice(source['test_file'], n_user, mr, [], [], n_group, train_index, 'r', dev)
    return ([loadData(d, batch, 1) for d in train], [loadData(d, batch, 1, False) for d in test],
            loadData(total, batch, 1, False), train_index)
