"""B200 mirror of the reference's numerics module (method/utils.py).

Same names, argument meaning and return values as the reference for everything on the
hot path -- ``MF``, ``baseTrain``, ``baseTest``, ``computeNDCG``, ``computeDCG``,
``ot_cluster``, ``seed_all``, ``saveObject``/``loadObject`` -- but the arithmetic runs in
libultrare_b200.so (hand-written sm_100a kernels).  There is no CPU path: calling any of
these without a CUDA device raises.

Out of scope (SURVEY.md §2.1 rows 14-16): u2u/d2d regularisers, k-means/k-medoids/LPA
clusterers, plotting helpers -- none is reachable from main.py.
"""
from __future__ import annotations

import pickle
import time
from functools import wraps

import numpy as np
import torch
from torch import nn

from .. import kernels as kn

STD = 1  # reference utils.py:27


def seed_all(seed):
    """reference utils.py:21-25 (plus torch.manual_seed, SURVEY Appendix A6)."""
    np.random.seed(seed)
    torch.manual_seed(seed)
    if torch.cuda.is_available():
        torch.cuda.manual_seed(seed)


def _cuda_device(device=None) -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("ultrare_b200 needs a CUDA device: the hot path has no CPU implementation")
    if device is None or str(device) in ("cuda", "cpu"):
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device(device)


class MF(nn.Module):
    """reference utils.py:30-43: two embedding tables, N(0, STD) init, dot-product forward.

    The tables are created directly on the GPU.  ``generator`` makes the init reproducible
    (the reference draws from the unseeded default generator, SURVEY.md §0.5).
    """

    def __init__(self, n_user, n_item, k=16, device=None, generator=None, user_rows=None):
        super().__init__()
        self.k = k
        dev = _cuda_device(device)
        # user_rows: build only these rows of the user table (compact per-shard table, DESIGN.md);
        # the values are the same rows a full-table init would have produced.
        P = self._normal((n_user, k), dev, generator)
        if user_rows is not None:
            P = P.index_select(0, user_rows)
        Q = self._normal((n_item, k), dev, generator)
        self.user_mat = nn.Embedding(P.shape[0], k, _weight=P)
        self.item_mat = nn.Embedding(n_item, k, _weight=Q)
        self.user_mat.weight.requires_grad_(False)
        self.item_mat.weight.requires_grad_(False)

    @classmethod
    def from_weights(cls, P, Q, device=None):
        """Model with given tables (parity runs inject the reference's initial weights)."""
        dev = _cuda_device(device)
        self = cls.__new__(cls)
        nn.Module.__init__(self)
        P = torch.as_tensor(P, dtype=torch.float32).to(dev).contiguous().clone()
        Q = torch.as_tensor(Q, dtype=torch.float32).to(dev).contiguous().clone()
        self.k = P.shape[1]
        self.user_mat = nn.Embedding(P.shape[0], self.k, _weight=P)
        self.item_mat = nn.Embedding(Q.shape[0], self.k, _weight=Q)
        self.user_mat.weight.requires_grad_(False)
        self.item_mat.weight.requires_grad_(False)
        return self

    @classmethod
    def wrap(cls, P, Q):
        """Model over existing device tensors (no copy): views into a batch allocation."""
        self = cls.__new__(cls)
        nn.Module.__init__(self)
        self.k = P.shape[1]
        self.user_mat = nn.Embedding(P.shape[0], self.k, _weight=P)
        self.item_mat = nn.Embedding(Q.shape[0], self.k, _weight=Q)
        self.user_mat.weight.requires_grad_(False)
        self.item_mat.weight.requires_grad_(False)
        return self

    @staticmethod
    def _normal(shape, dev, generator):
        """N(0, STD) (reference utils.py:38-40).  A host generator gives device-independent values;
        a CUDA generator (or None) draws on the GPU."""
        if generator is not None and generator.device.type == 'cpu':
            return torch.empty(shape, dtype=torch.float32).normal_(0.0, STD, generator=generator).to(dev)
        return torch.empty(shape, dtype=torch.float32, device=dev).normal_(0.0, STD, generator=generator)

    def init_weight(self, generator=None):
        dev = self.user_mat.weight.device
        self.user_mat.weight.data.copy_(self._normal(tuple(self.user_mat.weight.shape), dev, generator))
        self.item_mat.weight.data.copy_(self._normal(tuple(self.item_mat.weight.shape), dev, generator))

    def forward(self, uid, iid):
        dev = self.user_mat.weight.device
        inter = kn.pack_interactions(uid.cpu().numpy(), iid.cpu().numpy(), np.zeros(len(uid)), dev)
        score, _ = kn.ensemble_score([self.user_mat.weight.data], [self.item_mat.weight.data], inter)
        return score


class FusedSGD:
    """Stands where the reference builds optim.SGD + StepLR (scratch.py:65-69).

    Holds the hyper-parameters; momentum buffers, gradient scratch and the step counter live
    in the ShardState the first ``baseTrain`` call binds to the (loader, model) pair.
    loss: 'mse' (the reference's squared rating error) or 'bpr' (pairwise ranking, kernels.ShardBatch(loss='bpr')).
    """

    def __init__(self, model: MF, lr=1e-3, weight_decay=0.1, momentum=0.9, lr_decay=0.95, lr_step=50,
                 epochs=1, perm_seed=42, shard_id=0, loss='mse'):
        self.model = model
        self.loss = loss
        self.lr, self.weight_decay, self.momentum = lr, weight_decay, momentum
        self.lr_decay, self.lr_step, self.epochs = lr_decay, lr_step, epochs
        self.perm_seed, self.shard_id = perm_seed, shard_id
        self.batch_obj = None
        self.epoch = 0

    def bind(self, loader):
        if self.batch_obj is None:
            dev = self.model.user_mat.weight.device
            st = kn.ShardState(loader.dataset.records(dev), self.model.user_mat.weight.data,
                               self.model.item_mat.weight.data, self.epochs, shard_id=self.shard_id,
                               perm_seed=self.perm_seed, perm=loader.explicit_perm(dev, self.epochs))
            self.batch_obj = kn.ShardBatch([st], self.model.k, loader.batch_size, self.lr, self.lr_decay,
                                           self.lr_step, self.weight_decay, self.momentum, loss=self.loss)
        return self.batch_obj


def baseTrain(dataloader, model, loss_fn, is_rmse, opt, device, verbose, var='nor', attr=[]):
    """One training epoch (reference utils.py:46-111, var='nor'); returns (train_loss, rmse).

    ``opt`` is a FusedSGD; ``loss_fn`` is accepted for signature parity (the kernel computes
    MSELoss(reduction='sum'), scratch.py:45).  One persistent launch per call, one sync for
    the epoch's loss (the reference syncs every batch, utils.py:82).  With ``opt.loss == 'bpr'`` both values are
    the epoch's mean BPR loss, sum softplus(-x) / n.
    """
    assert var in ['nor'], "only the 'nor' path exists in the reference's reachable code"
    assert is_rmse, "the MF path uses MSELoss (scratch.py:44-46)"
    sb = opt.bind(dataloader)
    st = sb.shards[0]
    ep = opt.epoch
    if ep >= sb.epochs:
        raise RuntimeError("baseTrain called for more epochs than the optimiser was sized for")
    sb.train((ep + 1) * st.steps_per_epoch(sb.hp.batch))
    opt.epoch += 1
    sse = float(st.sse[ep].item())
    if opt.loss == 'bpr':
        train_loss = sse / max(1, st.n)
    else:
        train_loss = float(np.sqrt(sse / max(1, st.n)))
    return train_loss, train_loss


def base_test_device(dataloader, models):
    """The evaluation kernels of baseTest queued on the stream, no synchronisation: returns the device tensor
    fp64 [4] = (sum of squared errors, sum of NDCG@10, sum of HR@10, users) and the number of test rows."""
    dev = models[0].user_mat.weight.device
    ds = dataloader.dataset
    inter = ds.records(dev)
    vals = torch.zeros(4, dtype=torch.float64, device=dev)      # one clear, both kernels add into their slice
    score, _ = kn.ensemble_score([m.user_mat.weight.data for m in models],
                                 [m.item_mat.weight.data for m in models], inter, sse=vals[0:1])
    order, seg = ds.segments(dev, models[0].user_mat.weight.shape[0])
    kn.rank_metrics(inter, score, seg, order, out=vals[1:4])
    return vals, len(ds)


def base_test_values(vals, size):
    """(rmse, ndcg, hr) from the four sums of base_test_device (host values)."""
    rmse = float(np.sqrt(vals[0] / max(1, size)))
    users = max(vals[3], 1.0)
    return rmse, float(vals[1] / users), float(vals[2] / users)


def baseTest(dataloader, models, loss_fn, device, verbose, top_k=10):
    """Ensemble evaluation (reference utils.py:115-187); returns (rmse, ndcg, hr).

    Tie order of the per-user top-10: descending value, later index first (SURVEY.md H7).
    """
    assert top_k == kn._lib.URE_TOP_K
    vals, size = base_test_device(dataloader, models)
    rmse, ndcg, hr = base_test_values(kn.download_many([vals])[0], size)
    if verbose == 2:
        print(f'Test - RMSE: {rmse:>.4f}, NDCG: {ndcg:>.3f}, HR: {hr:>.3f}')
    return rmse, ndcg, hr


def _exclude_records(exclude, device):
    """Training records whose items are excluded: None, an int32 [n, 4] records tensor, a dataset / DataLoader, or a
    list of them; returns a records tensor, a list of them, or None."""
    if exclude is None:
        return None
    if isinstance(exclude, torch.Tensor):
        if exclude.dim() != 2 or exclude.shape[1] != 4 or exclude.dtype != torch.int32:
            raise ValueError("exclude: a records tensor must be int32 [n, 4]")
        return exclude.to(device)
    if isinstance(exclude, (list, tuple)):
        return [_exclude_records(e, device) for e in exclude]
    ds = getattr(exclude, 'dataset', exclude)
    return ds.records(device)


def _request_users(users, n_user, device):
    """The requested user ids as an int32 device tensor (all users when None); ids outside [0, n_user) raise."""
    if users is None:
        return torch.arange(n_user, dtype=torch.int32, device=device)
    u = torch.as_tensor(users).to(device=device, dtype=torch.int32).reshape(-1)
    if u.numel() > 0 and (int(u.min()) < 0 or int(u.max()) >= n_user):
        raise ValueError(f"recommend: user ids must lie in [0, {n_user})")
    return u


def recommend_from_tables(P, S, n_models, users=None, top_n=10, exclude=None):
    """(items int32 [m, top_n], scores fp32 [m, top_n]) of the ensemble mean (1/n_models) P[u].S[i], S the sum of the
    models' item tables; see ``recommend``."""
    dev = P.device
    u = _request_users(users, P.shape[0], dev)
    recs = _exclude_records(exclude, dev)
    seen = kn.seen_lists(recs, P.shape[0], S.shape[0]) if recs is not None else None
    return kn.recommend_topn(P, S, u, top_n, 1.0 / n_models, seen)


def recommend(models, users=None, top_n=10, exclude=None):
    """Top-N items per user over the whole catalogue: (items int32 [m, top_n], scores fp32 [m, top_n]) on the device.

    score(u, i) = (1/K) sum_k P_k[u].Q_k[i] (the baseTest ensemble mean) for the K models, which must share one user
    table (every SISA shard model does after the merge; a single model is a list of one).  Lists are sorted by score,
    ties to the smaller item id, and padded with item -1 / score -inf when fewer than top_n items are eligible.
    ``users``: ids in any order, duplicates allowed (None: every user).  ``exclude``: items a user has seen and must
    not be shown -- None, an int32 [n, 4] records tensor, a dataset or DataLoader, or a list of them.
    """
    if not models:
        raise ValueError("recommend: no models")
    P = models[0].user_mat.weight.data
    for m in models[1:]:
        Pm = m.user_mat.weight.data
        if Pm.data_ptr() != P.data_ptr() and (Pm.shape != P.shape or not torch.equal(Pm, P)):
            raise ValueError("recommend: the models' user tables differ (only ensembles sharing one user table are "
                             "supported)")
    S = kn.item_sum([m.item_mat.weight.data for m in models])
    return recommend_from_tables(P, S, len(models), users, top_n, exclude)


COMBINE_RIDGE = 1e-6     # lambda_g = COMBINE_RIDGE * tr(X_g^T X_g) / K: keeps the solve regular, the intercept free


class Combination:
    """A fitted combination of K shard models: per owner group g, s(u, i) = b[g] + sum_k w[g, k] P[u].Q_k[i].

    w fp64 [K, K], b fp64 [K] (host); T fp32 [K + 1, n_item, d] and b_slot fp32 [K + 1] on the device, where
    T[g] = sum_k w[g, k] Q_k and the last slot is the mean combination (w = 1/K, b = 0) that scores users in no group;
    gram: the fp64 kernel output the fit was solved from."""

    def __init__(self, w, b, T, b_slot, gram):
        self.w, self.b, self.T, self.b_slot, self.gram = w, b, T, b_slot, gram

    def table(self):
        """fp64 [K, K + 1]: row g = (w_g, b_g), the layout of combine.npy."""
        return np.concatenate([self.w, self.b[:, None]], axis=1)


def solve_combination(gram, K):
    """(w fp64 [n_groups, K], b fp64 [n_groups]) from ure_combine_gram's rows: per group the ridge least squares
    min sum (b + w.x - r)^2 + lambda ||w||^2, lambda = COMBINE_RIDGE * tr(X^T X) / K, the intercept not penalised,
    solved in float64 from the (K+1) x (K+1) normal equations.  A group without rows gets the mean (w = 1/K, b = 0)."""
    gram = np.asarray(gram, dtype=np.float64).reshape(-1, kn.combine_gram_entries(K))
    iu = np.triu_indices(K + 1)
    U = len(iu[0])
    w = np.full((gram.shape[0], K), 1.0 / K)
    b = np.zeros(gram.shape[0])
    for g, row in enumerate(gram):
        if row[-1] == 0:
            continue
        A = np.zeros((K + 1, K + 1))
        A[iu] = row[:U]
        A = A + np.triu(A, 1).T
        lam = COMBINE_RIDGE * np.trace(A[:K, :K]) / K
        A[np.arange(K), np.arange(K)] += lam
        m = row[U:U + K + 1]
        try:
            th = np.linalg.solve(A, m)
        except np.linalg.LinAlgError:        # all features zero: no ridge either; the minimum-norm solution
            th = np.linalg.lstsq(A, m, rcond=None)[0]
        w[g], b[g] = th[:K], th[K]
    return w, b


def fit_combination(P, Q_list, inters):
    """Fit the per-group combination of the models (P, Q_k), k < K, on the training records of every owner group
    (inters[g]: int32 [n, 4] device records, one per group, g < K; after an unlearn, the retained rows).  The Gram
    comes from ure_combine_gram, the ridge solve and the fallbacks are solve_combination's, T from ure_item_wsum."""
    K = len(Q_list)
    if len(inters) != K:
        raise ValueError(f"fit_combination: {len(inters)} record lists for {K} models (one per owner group)")
    gram = kn.combine_gram(P, Q_list, inters)
    gram_h = kn.download_many([gram])[0]
    w, b = solve_combination(gram_h, K)
    return combination_from(w, b, Q_list, gram_h)


def combination_from(w, b, Q_list, gram):
    """The Combination of given weights (w fp64 [K, K], b fp64 [K]) over the item tables Q_list: T from
    ure_item_wsum, b_slot uploaded; what fit_combination builds after its solve, and what a loaded state rebuilds."""
    K = len(Q_list)
    dev = Q_list[0].device
    W = np.concatenate([w, np.full((1, K), 1.0 / K)]).astype(np.float32)
    T = kn.item_wsum(Q_list, kn.upload_array(W, dev))
    b_slot = kn.upload_array(np.append(b, 0.0).astype(np.float32), dev)
    return Combination(w, b, T, b_slot, gram)


def recommend_combined(P, comb, owner, users, top_n=10, exclude=None, keep=None):
    """Top-N lists under a fitted Combination: (items int32 [m, top_n], scores fp32 [m, top_n]).  One ure_topn call per
    owner group among the requested users (T[g], scale 1), b[g] added to the returned scores but not to the -inf
    padding; users in no group use the mean slot.  The seen lists are built once.  keep: bool [m] device mask of the
    rows to compute; the other rows stay zero (several GPUs: each rank fills the rows of the groups it holds)."""
    dev = P.device
    u = _request_users(users, P.shape[0], dev)
    recs = _exclude_records(exclude, dev)
    seen = kn.seen_lists(recs, P.shape[0], comb.T.shape[1]) if recs is not None else None
    mean_slot = comb.T.shape[0] - 1
    o = owner[u.long()]
    slot = torch.where(o >= 0, o, torch.full_like(o, mean_slot))
    if keep is not None:
        slot = torch.where(keep, slot, torch.full_like(slot, -1))
    slot_h = slot.cpu().numpy()
    items = torch.zeros((u.shape[0], top_n), dtype=torch.int32, device=dev)
    scores = torch.zeros((u.shape[0], top_n), dtype=torch.float32, device=dev)
    for g in np.unique(slot_h[slot_h >= 0]).tolist():
        pos = torch.from_numpy(np.flatnonzero(slot_h == g)).to(dev)
        it, sc = kn.recommend_topn(P, comb.T[g], u[pos], top_n, 1.0, seen)
        items[pos] = it
        scores[pos] = torch.where(it >= 0, sc + comb.b_slot[g], sc)
    return items, scores


def topn_metrics(items, users, test_data, top_n):
    """Full-catalogue HR@N / Recall@N / NDCG@N of top-N lists (``recommend``'s items for ``users``; None = every user,
    row u for user u) against ``test_data`` (dataset, DataLoader or records tensor): relevant items are a user's
    distinct test items with normalised rating >= 4/5 (utils.py:175,180), users without one are not counted.
    Returns dict(hr, recall, ndcg, users) with the three metrics averaged over the counted users."""
    items = items[:, :top_n]
    dev = items.device
    inter = _exclude_records(test_data, dev)
    inter = kn._records_of(inter) if isinstance(inter, list) else inter
    u = torch.arange(items.shape[0], dtype=torch.int32, device=dev) if users is None else \
        torch.as_tensor(users).to(device=dev, dtype=torch.int32).reshape(-1)
    n_user = 1 + max(int(u.max()) if u.numel() else 0, int(inter[:, 0].max()) if inter.shape[0] else 0)
    vals = kn.download_many([kn.topn_metrics(items, u, inter, n_user)])[0]
    cnt = max(vals[3], 1.0)
    return dict(hr=float(vals[0] / cnt), recall=float(vals[1] / cnt), ndcg=float(vals[2] / cnt), users=int(vals[3]))


def computeNDCG(r, top_k):
    """reference utils.py:190-207 (host helper; the GPU path is ure_rank_metrics)."""
    r = np.asarray(r, dtype=np.float64)
    n = len(r)
    if n == 0:
        return 0
    r = np.concatenate([r, np.zeros(top_k - n)])
    assert len(r) == top_k
    return computeDCG(r) / computeDCG(np.ones(top_k))


def computeDCG(r):
    """reference utils.py:209-210."""
    return r[0] + np.sum(r[1:] / np.log2(np.arange(2, len(r) + 1)))


def saveObject(filename, obj):
    with open(filename + '.pkl', 'wb') as output:
        pickle.dump(obj, output, pickle.HIGHEST_PROTOCOL)


def loadObject(filename):
    with open(filename + '.pkl', 'rb') as f:
        return pickle.load(f)


def timefn(fn):
    """reference utils.py:616-626."""
    @wraps(fn)
    def measure_time(*args, **kwargs):
        t1 = time.time()
        result = fn(*args, **kwargs)
        t2 = time.time()
        print(f"@time: {t2 - t1: .5f} s")
        return result
    return measure_time


# Sinkhorn epsilon schedule, relative to the mean nearest-centroid cost (inertia / n):
# (eps_rel, iterations).  The reference's `lam = 1e-3` was never a regulariser (it lands in
# ot.emd's numItermax slot, SURVEY.md §0.2); eps -> 0 recovers its exact plan.
SINKHORN_SCHEDULE = ((1.0, 10), (0.3, 20), (0.1, 30), (0.03, 60), (0.01, 120))
# A stage ends early once the relative column-marginal error max_j |colsum_j*k - 1| drops below this; the
# fixed schedule itself only reaches ~3e-5 at its last stage, so nothing is lost.
SINKHORN_TOL = 2e-5
# With the balanced rounding behind it Sinkhorn only has to get the group sizes NEAR n/k: whatever the potentials, the
# argmax labels are the minimum-cost assignment for their own sizes, and the rounding moves the surplus users along
# shortest augmenting paths to the exact balanced optimum.  Measured at ml1m size (tools/prof_ot_small.py): the same
# labels for every tolerance from 2e-5 to 1e-2, 8.9 -> 5.9 ms for the ten outer iterations at 1e-3.
SINKHORN_TOL_BALANCED = 1e-3
# Outer iterations after the first start from the previous potentials (the fixed point at a given eps does
# not depend on the start) and run only the last WARM_STAGES stages of the schedule.  The column sums are kept in
# the log domain (csrc/ot_sinkhorn.cu), so potentials that are stale by hundreds of eps after a large centroid move
# recover in one iteration instead of underflowing.
SINKHORN_WARM_STAGES = 2
# Balanced rounding (csrc/ot_balance.cu): at most this many augmenting paths per outer iteration
BALANCE_MAX_AUGMENTATIONS = 1 << 14


def ot_cluster_device(X, k, max_iters=10, schedule=SINKHORN_SCHEDULE, centroid0=None, device=None, dist=None,
                      tol=None, warm_start=True, balance=True):
    """Balanced OT clustering on the GPU; returns (inertia, label int64 ndarray, centroid, n_outer).

    Per outer iteration (reference utils.py:635-654): cost matrix (tcgen05), Sinkhorn potentials, argmax labels,
    then -- ``balance`` -- the balanced rounding that moves the few users the entropic plan leaves on the wrong side
    along shortest augmenting paths, so that every group holds floor(n/k)..ceil(n/k) users at minimum cost, which is
    what the reference's exact ``ot.emd`` plan gives (utils.py:644-647); centroids from the final labels.

    With ``dist`` (ultrare_b200.dist.Dist, world_size > 1) X is this rank's row block, the column marginals /
    centroid sums are all-reduced and the rounding is skipped (the cost rows live on different GPUs).
    """
    dev = _cuda_device(device)
    X = np.ascontiguousarray(X, dtype=np.float32)
    n_local, d = X.shape
    sharded = dist is not None and dist.world > 1
    n = dist.sum_int(n_local) if sharded else n_local
    if centroid0 is None:
        if sharded:
            raise ValueError("distributed ot_cluster needs explicit initial centroids")
        centroid = X[np.random.choice(n, size=k, replace=False)]           # reference utils.py:632
    else:
        centroid = np.asarray(centroid0, dtype=np.float32)
    if d > 128:
        raise ValueError("ot_cluster: embedding dimension > 128 is not supported by the cost kernel")
    d_pad = next(v for v in (8, 16, 32, 64, 128) if v >= d)      # zero columns do not change the cost
    Xp = np.zeros((n_local, d_pad), dtype=np.float32)
    Xp[:, :d] = X
    Xd = kn.upload_table(Xp, dev)

    def cost(centroid):
        Cp = np.zeros((k, d_pad), dtype=np.float32)
        Cp[:, :d] = centroid
        return kn.cost_matrix(Xd, kn.upload_array(Cp, dev), want_inertia=True)     # utils.py:637-638

    def new_centroid(sums_h, cnt_h):
        return (sums_h[:, :d] / cnt_h[:, None]).astype(np.float32)

    return _ot_outer_loop(n, k, centroid, cost, lambda label: kn.centroid_sums(Xd, label, k), new_centroid,
                          max_iters, schedule, dist if sharded else None, tol, warm_start, balance)


def sparse_records(X):
    """int32 [nnz, 4] records (user, item, fp32 value bits, 0) of the stored entries of a SciPy sparse matrix, duplicates
    included: what ot_cluster_sparse_device uploads for kernels.sparse_orders."""
    coo = X.tocoo()
    rec = np.zeros((coo.nnz, 4), dtype=np.int32)
    rec[:, 0], rec[:, 1] = coo.row, coo.col
    rec[:, 2] = np.ascontiguousarray(coo.data, dtype=np.float32).view(np.int32)
    return rec


def ot_cluster_sparse_device(X, k, max_iters=10, schedule=SINKHORN_SCHEDULE, centroid0=None, device=None, dist=None,
                             tol=None, warm_start=True, balance=True):
    """``ot_cluster_device`` with the users' rows of a SciPy sparse matrix X [n, n_item] as the points (the reference's
    'rating-ot' grouping, group.py on readSparseMat); returns (inertia, label int64 ndarray, centroid fp32 [k, n_item],
    n_outer).  The nonzeros are uploaded once and ordered by user and by item on the device (kernels.sparse_orders);
    per outer iteration the cost matrix comes from ure_sparse_cost and the centroid sums from ure_sparse_centroid_sums,
    the rest of the loop is ot_cluster_device's.  Duplicate (user, item) entries count as their sum, as in SciPy; a
    user without entries is the zero row.  2 <= k <= 128 (the balanced rounding's limit).  One GPU: the grouping runs
    on rank 0 and is broadcast (config.Instance._group_index), so ``dist`` with several ranks raises."""
    import scipy.sparse as sp
    if not sp.issparse(X):
        raise TypeError("ot_cluster_sparse_device: X must be a SciPy sparse matrix")
    if dist is not None and dist.world > 1:
        raise ValueError("ot_cluster_sparse_device runs on one GPU (cluster on rank 0 and broadcast the labels)")
    if not 2 <= k <= kn._lib.URE_SPARSE_OT_MAX_K:
        raise ValueError(f"ot_cluster_sparse_device: k={k} outside 2 .. {kn._lib.URE_SPARSE_OT_MAX_K}")
    dev = _cuda_device(device)
    X = sp.csr_matrix(X, dtype=np.float32)
    n, n_item = X.shape
    if k > n:
        raise ValueError(f"ot_cluster_sparse_device: k={k} > {n} users")
    if centroid0 is None:
        centroid = X[np.random.choice(n, size=k, replace=False)].toarray()  # reference utils.py:632
    else:
        centroid = np.asarray(centroid0, dtype=np.float32)
    csr, csc = kn.sparse_orders(kn.upload_table(sparse_records(X), dev), n, n_item)
    kp = kn.kpad_for(k)

    def cost(centroid):
        Ct = np.zeros((n_item, kp), dtype=np.float32)
        Ct[:, :k] = centroid.T
        cnorm = np.square(centroid.astype(np.float64)).sum(axis=1)
        return kn.sparse_cost(csr, kn.upload_array(Ct, dev), kn.upload_array(cnorm, dev), k, want_inertia=True)

    def new_centroid(sums_h, cnt_h):
        return (sums_h[:, :k].T / cnt_h[:, None]).astype(np.float32)

    return _ot_outer_loop(n, k, np.asarray(centroid, dtype=np.float32), cost,
                          lambda label: kn.sparse_centroid_sums(csc, label, k), new_centroid,
                          max_iters, schedule, None, tol, warm_start, balance)


def _ot_outer_loop(n, k, centroid, cost, centroid_sums, new_centroid, max_iters, schedule, dist, tol, warm_start,
                   balance):
    """The outer loop both ot_cluster paths share (reference utils.py:635-654).  cost(centroid) -> (M [n_local, kpad],
    fp64 inertia tensor); centroid_sums(label) -> (sums, counts [k]) device tensors; new_centroid(sums, counts) -> the
    next centroids from their host copies.  dist: a Dist with several ranks (rows sharded), or None."""
    sharded = dist is not None
    balance = balance and not sharded and 1 < k <= 128
    if tol is None:
        tol = SINKHORN_TOL_BALANCED if balance else SINKHORN_TOL
    label = None
    g = None
    inertia = 0.0
    it = 0
    for it in range(1, max_iters + 1):
        M, inert = cost(centroid)
        if sharded:
            dist.all_reduce(inert)
        inertia = float(kn.download_many([inert])[0][0])
        scale = max(inertia / n, 1e-30)
        warm = warm_start and it > 1
        sched = [(e * scale, i) for e, i in (schedule[-SINKHORN_WARM_STAGES:] if warm else schedule)]
        if not sharded:
            g = kn.sinkhorn(M, k, sched, g=g if warm else None, tol=tol)    # replaces ot.emd, utils.py:641-644
        else:
            g = kn.sinkhorn_sharded(M, k, sched, dist, n, g=g if warm else None)
        label, _, cnt = kn.assign_centroids(M, k, g, None)                  # utils.py:647 (argmax of the plan row)
        status = kn.balance_labels(M, k, label, cnt, BALANCE_MAX_AUGMENTATIONS) if balance else None
        sums, cnt = centroid_sums(label)                                    # utils.py:648
        if sharded:
            dist.all_reduce(sums)
            dist.all_reduce(cnt)
        got = kn.download_many([sums, cnt, g] + ([status] if balance else []))        # the iteration's one sync
        sums_h, cnt_h, g_h = got[0], got[1], got[2]
        if not np.isfinite(g_h).all():
            raise RuntimeError(f"ot_cluster: Sinkhorn potentials are not finite ({g_h}); non-finite embedding or "
                               f"centroid?")
        if (cnt_h[:k] == 0).any():
            raise RuntimeError(f"ot_cluster: empty group (sizes {cnt_h[:k].tolist()}); the plan is degenerate")
        if balance and (got[3][1] != 0 or got[3][2] != 0):
            import warnings
            warnings.warn(f"ot_cluster: balanced rounding stopped early ({int(got[3][0])} augmentations, "
                          f"{int(got[3][1])} users still to move); group sizes {cnt_h[:k].tolist()}")
        nxt = new_centroid(sums_h, cnt_h)
        if np.allclose(centroid, nxt):                                       # utils.py:651
            break
        centroid = nxt
    return np.float32(inertia), label.cpu().numpy().astype(np.int64), centroid, it


@timefn
def ot_cluster(X, k, max_iters=10):
    """reference utils.py:628-656: returns (inertia, label).  X: a dense [n, d] embedding, or a SciPy sparse matrix of
    the users' rating rows ('rating-ot', ot_cluster_sparse_device)."""
    import scipy.sparse as sp
    run = ot_cluster_sparse_device if sp.issparse(X) else ot_cluster_device
    inertia, label, _, _ = run(X, k, max_iters)
    print(f'{inertia:.3f}', end=' ')
    return inertia, label
