"""B200 mirror of the reference's read.py: shard materialisation and (device) loaders.

``readRating`` / ``sort_group`` keep the reference's signature and return values
(read.py:9-106) with its defects resolved as SURVEY.md Appendix A lists (A8: no dependence
on 'ml1m' appearing in the path, A9: no debug prints).  ``RatingData`` / ``loadData``
(read.py:108-133) keep the attributes the rest of the code touches (``.dataset.users/
items/ratings``, ``len``), but a loader is a thin descriptor: batches are never
materialised on the host -- the training kernel walks the shard's device-resident records
in the epoch's permutation order (the per-sample ``__getitem__`` + collate of the
reference is its #1 cost, SURVEY.md §8 a7).
"""
from __future__ import annotations

import numpy as np
import pandas as pd
import torch

from . import kernels as kn


def _pair_keys(del_rating):
    """Deleted ratings as sorted unique int64 keys (int(user) << 32) | int(item), or None when there are none.
    del_rating: array-like [n, >= 2] of (user, item, ...); negative ids raise ValueError."""
    if len(del_rating) == 0:
        return None
    p = np.asarray(del_rating)
    if p.ndim != 2 or p.shape[1] < 2:
        raise ValueError(f"del_rating must be [n, >= 2] (user, item, ...), got shape {p.shape}")
    p = p[:, :2].astype(np.int64)
    if (p < 0).any():
        raise ValueError("del_rating: user and item ids must be non-negative")
    if (p >= 2 ** 31).any():
        raise ValueError("del_rating: user and item ids must be below 2^31")
    return np.unique((p[:, 0] << 32) | p[:, 1])


def _row_keys(ratings):
    """The keys of _pair_keys for every row of the ratings table (ids truncated to int, as the partition kernel does)."""
    u = ratings[0].values.astype(np.int64)
    i = ratings[1].values.astype(np.int64)
    return (u << 32) | (i & 0xFFFFFFFF)


def readRating(dir, n_user, max_rating=5, del_user=[], del_rating=[], n_group=1, group_index=[], sort='r'):
    """reference read.py:9-70.  Returns (rating_lists [n_group] of float64 [3,n_g], group_index).
    del_rating: (user, item) pairs whose rows are dropped (interaction-level unlearning); the group order is that
    of the unfiltered table."""
    if len(group_index) == 0:
        group_len = int(np.ceil(n_user / n_group))
        org_index = np.arange(n_user).tolist()
        if n_group == 1:
            group_index = [org_index]
        else:
            np.random.seed(0)
            np.random.shuffle(org_index)
            group_index = [org_index[i * group_len:(i + 1) * group_len] for i in range(n_group)]

    ratings = dir if isinstance(dir, pd.DataFrame) else pd.read_csv(dir, header=None, sep=',')
    users = ratings[0].values
    vals = ratings.values

    if sort in ['d', 'a']:
        sorted_index = sort_group(order='a', group_index=group_index, var='count', ratings0=users)
        group_index = [group_index[i] for i in sorted_index]

    # owner map: one pass instead of K np.in1d scans (a user belongs to the first group listing it)
    owner = np.full(max(n_user, int(users.max()) + 1 if len(users) else 0), -1, dtype=np.int64)
    for g in range(n_group - 1, -1, -1):
        owner[np.asarray(group_index[g], dtype=np.int64)] = g
    deleted = np.zeros(len(owner), dtype=bool)
    if len(del_user):
        deleted[np.asarray(list(del_user), dtype=np.int64)] = True
    row_owner = np.where(deleted[users.astype(np.int64)], -1, owner[users.astype(np.int64)])
    del_keys = _pair_keys(del_rating)
    if del_keys is not None:
        row_owner = np.where(np.isin(_row_keys(ratings), del_keys), -1, row_owner)

    rating_lists = []
    for g in range(n_group):
        ratings_group = vals[row_owner == g].T.astype(np.float64).copy()
        if ratings_group.size == 0:
            ratings_group = np.zeros((3, 0), dtype=np.float64)
        ratings_group[2] /= max_rating
        rating_lists.append(ratings_group)
    return rating_lists, group_index


def readRatingDevice(dir, n_user, max_rating=5, del_user=[], del_rating=[], n_group=1, group_index=[], sort='r',
                     device='cuda'):
    """``readRating`` (reference read.py:9-70) with the row filter and the group split ON the device.

    The CSV is parsed on the host (pandas, as in the reference) and uploaded ONCE; one stable partition kernel
    (ure_partition_interactions) then does what read.py:36-68 does with K np.in1d scans.  Returns
    (datasets [n_group] of device-backed ``RatingData`` -- same rows, same row order as readRating's arrays --,
    group_index, total) where ``total`` is the RatingData of all groups back to back (config.py:144-148's hstack).
    del_rating: (user, item) pairs whose rows the same partition drops (ure_partition_interactions_del, with the
    per-user deleted-item lists of kernels.deletion_lists).
    """
    if len(group_index) == 0:                 # read.py:13-26, same RNG calls as readRating
        group_len = int(np.ceil(n_user / n_group))
        org_index = np.arange(n_user).tolist()
        if n_group == 1:
            group_index = [org_index]
        else:
            np.random.seed(0)
            np.random.shuffle(org_index)
            group_index = [org_index[i * group_len:(i + 1) * group_len] for i in range(n_group)]
    ratings = dir if isinstance(dir, pd.DataFrame) else pd.read_csv(dir, header=None, sep=',')
    users = ratings[0].values
    if sort in ['d', 'a']:
        sorted_index = sort_group(order='a', group_index=group_index, var='count', ratings0=users)
        group_index = [group_index[i] for i in sorted_index]
    n_map = max(n_user, int(users.max()) + 1 if len(users) else 0)
    owner = np.full(n_map, -1, dtype=np.int32)
    for g in range(n_group - 1, -1, -1):      # a user belongs to the first group that lists it
        owner[np.asarray(group_index[g], dtype=np.int64)] = g
    deleted = None
    if len(del_user):
        deleted = np.zeros(n_map, dtype=np.uint8)
        deleted[np.asarray(list(del_user), dtype=np.int64)] = 1
    del_keys = _pair_keys(del_rating)
    dev = torch.device(device)
    del_lists = None if del_keys is None else kn.deletion_lists(np.asarray(del_rating), n_map, dev)
    tab = np.empty((3, len(users)), dtype=np.float64)        # one cast pass per column (DataFrame.values would
    for j in range(3):                                       # first consolidate the mixed columns into a copy)
        tab[j] = ratings[j].values
    table = kn.upload_table(tab, dev)
    rec, off = kn.partition_interactions(table, max_rating, kn.upload_array(owner, dev),
                                         None if deleted is None else kn.upload_array(deleted, dev), n_group,
                                         del_lists=del_lists)
    off_h = off.cpu().numpy()
    src = (ratings, owner, deleted, float(max_rating), del_keys)
    datasets = [DeviceRatingData(rec[int(off_h[g]):int(off_h[g + 1])], src, (g, g + 1)) for g in range(n_group)]
    total = DeviceRatingData(rec[:int(off_h[n_group])], src, (0, n_group))
    return datasets, group_index, total


def sort_group(order='a', group_index=[], var='count', ratings0=[], dataset='ml1'):
    """reference read.py:73-106 (var='count': groups by ascending/descending rating count)."""
    assert var in ['count']
    ratings0 = np.asarray(ratings0).astype(np.int64)
    counts_per_user = np.bincount(ratings0, minlength=int(ratings0.max()) + 1 if len(ratings0) else 1)
    sort_value = []
    for index in group_index:
        idx = np.unique(np.asarray(index, dtype=np.int64))
        idx = idx[idx < len(counts_per_user)]
        sort_value.append(int(counts_per_user[idx].sum()))
    if order == 'a':
        return np.argsort(sort_value)
    return np.argsort(sort_value)[::-1]


def _mapped_key(device, tag, row_of):
    """Cache key of records whose user field went through `row_of`: the map's identity (storage address + version
    counter) is part of it, so a loader reused with ANOTHER grouping never returns rows of the previous one (the
    kernels index compact tables with these rows and do no bounds check)."""
    return (str(device), tag, int(row_of.data_ptr()), int(row_of._version), int(row_of.shape[0]))


# A torch.device: a RatingData built on a page-locked float64 [3, n] array (kernels.pinned_copy) starts its host -> device
# copy in the constructor, on the side stream -- the bytes travel while the caller still builds loaders, routes the
# deletions and lays out the batch; records() / records_mapped() / upload_many() then only pack.  None: off.
EAGER_UPLOAD_DEVICE = None


class RatingData:
    """reference read.py:108-124: users/items int, ratings float (already / max_rating)."""

    def __init__(self, rating_array):
        self._raw = rating_array              # [3, n]: uid, iid, rating / max_rating (float64, read.py:64-68)
        self._n = int(np.shape(rating_array[0])[0])
        self._cols = {}
        self._records = {}
        self._segments = {}
        self._maps = {}
        self._eager = kn.eager_upload(rating_array, EAGER_UPLOAD_DEVICE) if EAGER_UPLOAD_DEVICE is not None else None

    def _take_eager(self, device):
        """The columns an eager upload put on `device` (handed over once), or None."""
        e, self._eager = getattr(self, '_eager', None), None
        if e is None:
            return None
        want, have = torch.device(device), e[0].device
        same = want.type == have.type and (want.index is None or want.index == have.index)
        return e if same else None

    def _col(self, j, dtype):
        if j not in self._cols:               # the reference's eager casts (read.py:111-113), done on demand
            self._cols[j] = np.asarray(self._raw[j]).astype(dtype)
        return self._cols[j]

    users = property(lambda self: self._col(0, int))
    items = property(lambda self: self._col(1, int))
    ratings = property(lambda self: self._col(2, float))

    def __len__(self):
        return self._n

    def __getitem__(self, idx):
        return (torch.tensor(self.users[idx], dtype=torch.long),
                torch.tensor(self.items[idx], dtype=torch.long),
                torch.tensor(self.ratings[idx], dtype=torch.float32))

    def records(self, device) -> torch.Tensor:
        """int32 [n,4] ure_inter_t records resident on `device` (uploaded once)."""
        key = str(device)
        if key not in self._records:
            self._records[key] = kn.upload_interactions(self._raw, device, eager=self._take_eager(device))
        return self._records[key]

    def records_mapped(self, device, row_of: torch.Tensor, tag: str) -> torch.Tensor:
        """Records whose user field is row_of[user] (the row inside a compact per-shard user table);
        row_of: int32 tensor on `device`, applied by the pack kernel."""
        key = _mapped_key(device, tag, row_of)
        if key not in self._records:
            self._drop_mapped(device, tag)
            self._records[key] = kn.upload_interactions(self._raw, device, row_of, eager=self._take_eager(device))
            self._keep_map(key, row_of)
        return self._records[key]

    def _drop_mapped(self, device, tag):
        """Forget the records mapped through an earlier row_of (one mapped copy per (device, tag) is kept)."""
        for k in [k for k in self._records if isinstance(k, tuple) and k[:2] == (str(device), tag)]:
            del self._records[k]
            self._maps.pop(k, None)

    def _keep_map(self, key, row_of):
        self._maps[key] = row_of              # holds the tensor: its address cannot be reused while the key lives

    @staticmethod
    def upload_many(datasets, device, row_of=None, tag=None, defer=False):
        """records()/records_mapped() of several datasets at once: their host copies run in parallel.
        defer=True: the copies are started and a `finish()` callable is returned; the records are registered (and
        the uploads queued) when it is called."""
        key = str(device) if tag is None else _mapped_key(device, tag, row_of)
        for ds in datasets:
            if isinstance(ds, DeviceRatingData):
                ds.records(device) if tag is None else ds.records_mapped(device, row_of, tag)
        todo = [ds for ds in datasets if key not in ds._records]
        if not todo:
            return (lambda: None) if defer else None
        recs, fin = kn.upload_interactions_many([ds._raw for ds in todo], device, row_of, defer=True,
                                                eager=[ds._take_eager(device) for ds in todo])

        def finish():
            fin()
            for ds, rec in zip(todo, recs):
                if tag is not None:
                    ds._drop_mapped(device, tag)
                    ds._keep_map(key, row_of)
                ds._records[key] = rec

        if defer:
            return finish
        finish()

    DEVICE_SEGMENTS_MIN_ROWS = 1 << 18

    def segments(self, device, n_user=None):
        """(order or None, seg) device tensors of the per-user test segments (utils.py:151-161).  With n_user (an
        upper bound of the user ids: the rows of the user table) they are built on the device from the uploaded
        records, with no host pass over the data and no synchronisation; without it, by the host (file order)."""
        if n_user is not None and self._n < self.DEVICE_SEGMENTS_MIN_ROWS:
            n_user = None       # small sets: the host pass is hidden behind the training launch that precedes it
        key = str(device) if n_user is None else (str(device), int(n_user))
        if key not in self._segments:
            if n_user is not None:
                self._segments[key] = kn.user_segments_device(self.records(device), int(n_user))
            else:
                order, seg = kn.user_segments(self.users)
                self._segments[key] = (None if order is None else kn.upload_array(order, device),
                                       kn.upload_array(seg, device))
        return self._segments[key]


class DeviceRatingData(RatingData):
    """RatingData whose records were produced on the device by ``readRatingDevice``.  ``records()`` is the
    partition's output; the host columns (``users``/``items``/``ratings``, ``_raw``) are rebuilt on demand:
    ids from the records, the float64 ratings by the host filter of readRating (read.py:59-68).  src: (ratings table,
    owner map, deleted-user flags or None, max_rating[, deleted-rating keys of _pair_keys or None])."""

    def __init__(self, records, src, groups):
        self._dev = records
        self._src, self._groups = src, groups
        self._n = int(records.shape[0])
        self._cols, self._segments, self._maps = {}, {}, {}
        self._records = {str(records.device): records}

    def _rows(self):
        """Indices of this dataset's rows in the source table, in record order (host filter of read.py:59-62)."""
        if 'rows' not in self._cols:
            ratings, owner, deleted = self._src[:3]
            users = ratings[0].values.astype(np.int64)
            own = owner[users] if deleted is None else np.where(deleted[users] != 0, -1, owner[users])
            del_keys = self._src[4] if len(self._src) > 4 else None
            if del_keys is not None:
                own = np.where(np.isin(_row_keys(ratings), del_keys), -1, own)
            lo, hi = self._groups
            parts = [np.flatnonzero(own == g) for g in range(lo, hi)]
            self._cols['rows'] = np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)
        return self._cols['rows']

    @property
    def _raw(self):
        if 'raw' not in self._cols:
            ratings, max_rating = self._src[0], self._src[3]
            raw = np.stack([ratings[j].values[self._rows()].astype(np.float64) for j in range(3)])
            raw[2] /= max_rating
            self._cols['raw'] = raw
        return self._cols['raw']

    def _col(self, j, dtype):
        if j not in self._cols:               # host copies never wait for the device (it may be training)
            v = self._src[0][j].values[self._rows()]
            self._cols[j] = (v.astype(np.float64) / self._src[3] if j == 2 else v).astype(dtype)
        return self._cols[j]

    def records(self, device):
        key = str(device)
        if key not in self._records:
            d = torch.device(device)
            same = d.type == 'cuda' and (d.index is None or d.index == self._dev.device.index)
            self._records[key] = self._dev if same else self._dev.to(d)
        return self._records[key]

    def records_mapped(self, device, row_of, tag):
        key = _mapped_key(device, tag, row_of)
        if key not in self._records:
            self._drop_mapped(device, tag)
            self._records[key] = kn.remap_users(self.records(device).contiguous(), row_of)
            self._keep_map(key, row_of)
        return self._records[key]


class ShardLoader:
    """What ``loadData`` returns: the DataLoader arguments plus the dataset (read.py:127-133)."""

    def __init__(self, data, batch=30000, n_worker=24, shuffle=True, perms=None):
        self.dataset = data
        self.batch_size = batch
        self.n_worker = n_worker          # accepted for signature parity; there are no host workers
        self.shuffle = shuffle
        self.perms = perms                # optional explicit [epochs][n] visiting orders (parity runs)

    def __len__(self):
        return -(-len(self.dataset) // self.batch_size)

    def explicit_perm(self, device, epochs):
        n = len(self.dataset)
        if self.perms is not None:
            p = np.asarray(self.perms, dtype=np.int32)
            assert p.shape == (epochs, n), f"perms must be [{epochs},{n}]"
            return torch.from_numpy(np.ascontiguousarray(p)).to(device)
        if not self.shuffle:
            return torch.arange(n, dtype=torch.int32, device=device).repeat(epochs, 1)
        return None                       # keyed Feistel permutation inside the kernel


def loadData(data, batch=30000, n_worker=24, shuffle=True, perms=None):
    """reference read.py:127-133."""
    return ShardLoader(data, batch, n_worker, shuffle, perms)


def readSparseMat(dir, n_user, n_item, max_rating=5):
    """reference read.py:136-145; only its shape is used on the 'emb-ot' path (config.py:130)."""
    from scipy.sparse import coo_matrix
    ratings = pd.read_csv(dir, header=None, sep=',')
    row = ratings[0].astype(int).values
    col = ratings[1].astype(int).values
    val = ratings[2].astype(float).values / max_rating
    return coo_matrix((val, (row, col)), shape=(n_user, n_item), dtype=np.float32).tocsr()
