"""B200 mirror of the reference's SISA learner (method/sisa.py:7-118).

Same class, constructor and ``learn`` / ``unlearn`` / ``test`` signatures, same artefacts
(``model{i}.pth``, ``user_mat{i}.npy``, ``item_mat{i}.npy``, ``log{i}.npy``, ``log0.npy``).
What changes underneath:
  * the K shard trainings of sisa.py:33-36 / 86-89 (a sequential Python loop) become ONE
    persistent launch that trains every shard this GPU owns at once (kernels.ShardBatch);
  * deleted users are routed to their shards by an owner-map kernel (sisa.py:76-81 is a
    triple nested Python loop);
  * the owner-row merge (sisa.py:52-58, 107-113) is a gather kernel;
  * with torch.distributed initialised, shard s lives on rank s mod world and only the
    merged user table and the evaluation scores cross GPUs (ultrare_b200/dist.py).

``epoch_eval`` selects how much of the reference's per-epoch in-training evaluation
(scratch.py:83-128) is reproduced:
  'faithful'  every epoch of every shard is evaluated exactly as the reference does,
              including its quirk of ensembling the in-training model with
              ``self.model_list`` (scratch.py:83-86) -- from device snapshots taken at
              epoch boundaries, after the batched training.  Shard models keep the
              reference's full [n_user, k] user tables (the quirk reads non-owner rows).
  'final'     test_* of the last epoch of each shard only (earlier entries and total_* NaN);
  'none'      train_loss only.
In 'final' / 'none' mode each shard model stores only its owners' user rows (compact
table): rows a shard does not own never receive a gradient and are dropped by the merge, so
the merged table, the item tables and every final metric are unchanged.

``slices`` = R > 1 adds SISA's slicing (DESIGN.md §4): each shard's records are read slice-major (read.readRating /
readRatingDevice with n_slice=R), the shard trains in R stages of ``stage_epochs`` epochs each, stage r on slices
0..r-1 and starting from the weights after stage r-1, and the weights before every stage are kept as checkpoints with
the shard model.  An unlearn restarts each affected shard from the checkpoint before its first affected slice.

``save_state`` / ``load_state`` write and read the whole model (merged user table, item tables, checkpoints, fitted
combination, grouping, ledger of applied deletions) as a directory (DESIGN.md §4.10, method/sisa_state.py);
``apply_request`` unlearns a deletion request from it, minus what the ledger already holds.
"""
from __future__ import annotations

import json
import os
import time
import types
import warnings

import numpy as np
import torch
from torch import nn

from .. import dist as udist
from .. import kernels as kn
from .scratch import Scratch
from .utils import (_request_users, baseTest, base_test_device, base_test_values, fit_combination, recommend_combined,
                    recommend_from_tables)


def stage_epochs(epochs, slices):
    """Epochs of one slice stage, SISA's e' = max(1, ceil(2E / (R + 1))): the R stages then train about as many
    interactions as E unsliced epochs do.  R = 1 gives E."""
    return max(1, -(-2 * int(epochs) // (int(slices) + 1)))


class _Table:
    """Evaluation view of one model: just the two weight tensors."""

    def __init__(self, P, Q):
        self.user_mat = types.SimpleNamespace(weight=P)
        self.item_mat = types.SimpleNamespace(weight=Q)


class _RemoteModel:
    """Placeholder in model_list for a shard another GPU owns: the shared merged user table only."""

    def __init__(self, merged_param):
        self.user_mat = types.SimpleNamespace(weight=merged_param)
        self.item_mat = None


_OWNER_CACHE = {}


def _owner_maps(group_index, n_user, device):
    """owner[u] = group of user u (-1: none), row_of[u] = its row in the group's compact table; numpy + device
    copies, cached per group_index object (learn / unlearn / repeated requests reuse the same grouping)."""
    key = (id(group_index), n_user, str(device))
    hit = _OWNER_CACHE.get(key)
    if hit is not None and hit[0] is group_index:
        return hit[1:]
    owner = np.full(n_user, -1, dtype=np.int32)
    row_of = np.zeros(n_user, dtype=np.int32)
    for g in range(len(group_index) - 1, -1, -1):              # a user belongs to the FIRST group listing it
        ids = np.asarray(group_index[g], dtype=np.int64)
        owner[ids] = g
        row_of[ids] = np.arange(len(ids), dtype=np.int32)
    out = (owner, row_of, torch.from_numpy(owner).to(device), torch.from_numpy(row_of).to(device))
    if len(_OWNER_CACHE) > 8:
        _OWNER_CACHE.clear()
    _OWNER_CACHE[key] = (group_index,) + out
    return out


def _as_one_block(tensors):
    """The tensors as ONE [n, ...] view when they lie back to back in device memory in this order (the tables of a
    batch arena do), else None."""
    if not tensors:
        return None
    t0 = tensors[0]
    end = t0.data_ptr()
    for t in tensors:
        if t.data_ptr() != end or not t.is_contiguous() or t.dtype != t0.dtype or t.shape[1:] != t0.shape[1:]:
            return None
        end += t.numel() * t.element_size()
    rows = sum(int(t.shape[0]) for t in tensors)
    return torch.as_strided(t0, (rows,) + tuple(t0.shape[1:]), t0.stride())


def _local(models):
    return [m for m in models if m is not None and getattr(m, 'item_mat', None) is not None]


_EVAL_ROWS = {}
_WRITERS = []


def _writer_pool():
    if not _WRITERS:
        from concurrent.futures import ThreadPoolExecutor
        _WRITERS.append(ThreadPoolExecutor(max_workers=1))
    return _WRITERS[0]



def _eval_rows(recs, n_user):
    """(records, order, seg) of several resident test sets evaluated together; cached while the same device
    buffers are passed again (the cache holds them, so their addresses cannot be reused meanwhile)."""
    key = (tuple((r.data_ptr(), r.shape[0]) for r in recs), n_user)
    hit = _EVAL_ROWS.get(key)
    if hit is None:
        if len(recs) == 1:
            inter = recs[0]
        else:                              # back to back in one buffer: device-to-device copies, no kernel
            inter = torch.empty((sum(r.shape[0] for r in recs), 4), dtype=torch.int32, device=recs[0].device)
            o = 0
            for r in recs:
                inter[o:o + r.shape[0]].copy_(r, non_blocking=True)
                o += r.shape[0]
        order, seg = kn.user_segments_device(inter, n_user)
        _EVAL_ROWS.clear()                 # one entry: the resident test sets of the current run
        hit = _EVAL_ROWS[key] = (inter, order, seg, recs)
    return hit[0], hit[1], hit[2]


class Sisa(Scratch):
    def __init__(self, param={}, model_type='mf', n_group=5, group_index=[]):
        super(Sisa, self).__init__(param, model_type)
        self.n_group = n_group
        self.group_index = group_index
        self.model_list = []
        self.epoch_eval = os.environ.get('ULTRARE_EPOCH_EVAL', 'faithful')
        # multi-GPU final evaluation: None = shard the test rows over the ranks when test_data has as many rows
        # as the per-shard test sets together (it is their concatenation in Instance, config.py:144-148);
        # False = always score the whole of test_data on every rank (partial scores all-reduced)
        self.eval_sharded = None
        self._writers = []
        self.dist = udist.get()
        self._owner_np, self._row_of_np, self._owner, self._row_of = _owner_maps(group_index, self.n_user, self.device)
        self._group_rows = {}
        self.retrain_gid = set()
        self.timing = {}
        # how the final evaluation and recommend combine the shard models: 'mean' = the reference's (1/K) sum_k
        # P[u].Q_k[i]; 'fit' = the learned per-owner-group combination (utils.fit_combination), refitted on the
        # retained training rows after every learn / unlearn pass
        self.combine = 'mean'
        self.combination = None
        # SISA slicing: R stages per shard with a checkpoint before each (1 = unsliced, the reference's training)
        self.slices = 1
        # where the training data comes from (save_state records it; apply_request reads the retained data from it):
        # dict(dataset, train_file, test_file, max_rating, grouping, group_index) -- group_index is the grouping
        # before the reader's count sort ([]: the reader's uniform draw)
        self.source = None
        # the ledger: every deletion applied since the learn (sorted unique users, sorted unique (user, item) pairs)
        self.deleted_users = np.zeros(0, dtype=np.int64)
        self.deleted_pairs = np.zeros((0, 2), dtype=np.int64)
        self.requests = 0

    def _mode(self):
        if self.dist.world > 1 and self.epoch_eval == 'faithful':
            return 'final'          # the quirk needs every other shard's model on this GPU
        return self.epoch_eval

    def _rows(self, g):
        if g not in self._group_rows:
            self._group_rows[g] = torch.as_tensor(np.asarray(self.group_index[g], dtype=np.int64), device=self.device)
        return self._group_rows[g]

    # ------------------------------------------------------------------ evaluation
    def test(self, test_data, verbose, save_dir):
        """reference sisa.py:18-23."""
        if self._use_fit():
            rmse, ndcg, hr = self._combined_test(test_data, verbose)
        else:
            rmse, ndcg, hr = self._ensemble_test(test_data, verbose)
        log = {'total_rmse': rmse, 'total_ndcg': ndcg, 'total_hr': hr}
        if len(save_dir) > 0 and self.dist.rank == 0:
            np.save(save_dir + '/log0', log)
        self.final_log = log
        return log

    RECOMMEND_GATHER_BYTES = 256 << 20      # device memory of one chunk of gathered item tables (Sisa.recommend)

    def _item_sum_in_shard_order(self):
        """S = sum_k Q_k [n_item, d], summed in shard order k = 0 .. K-1 by ure_item_sum: the same bits at every world
        size.  On several GPUs the ranks all-gather their item tables chunk by chunk of item rows (shard s lives on rank
        s mod world) and every rank sums all K in order; an all-reduce of per-rank partial sums would associate the
        additions by rank and change the last bits of S, and with them near-tied lists."""
        K, world, rank = self.n_group, self.dist.world, self.dist.rank
        if world == 1:
            return kn.item_sum([self.model_list[s].item_mat.weight.data for s in range(K)])
        slots = -(-K // world)
        rows = max(1, min(self.n_item, self.RECOMMEND_GATHER_BYTES // (world * slots * self.k * 4)))
        part = torch.zeros((slots, rows, self.k), dtype=torch.float32, device=self.device)
        full = torch.empty((world * slots, rows, self.k), dtype=torch.float32, device=self.device)
        S = torch.empty((self.n_item, self.k), dtype=torch.float32, device=self.device)
        mine = list(range(rank, K, world))
        for r0 in range(0, self.n_item, rows):
            n = min(self.n_item, r0 + rows) - r0
            for j, s in enumerate(mine):
                part[j, :n].copy_(self.model_list[s].item_mat.weight.data[r0:r0 + n])
            self.dist.all_gather_into(full, part)
            S[r0:r0 + n].copy_(kn.item_sum([full[(s % world) * slots + s // world, :n] for s in range(K)]))
        return S

    def recommend(self, users=None, top_n=10, exclude=None):
        """Top-N items per requested user from the ensemble of ``model_list`` (see utils.recommend): (items int32
        [m, top_n], scores fp32 [m, top_n]) on the device, the same on every rank.  ``exclude``: the seen items to leave
        out (records, dataset, DataLoader or a list of them, e.g. the shards' training loaders).

        The item tables are summed in shard order whatever the number of GPUs (_item_sum_in_shard_order), so the
        result is the same bit for bit on one GPU and on several.  With several GPUs each rank recommends for the
        requested users whose owner shard it holds (users in no group: rank 0), because it holds those shards' training
        records, and the rows, placed by request position into zero-filled outputs, are all-reduced (every row has one
        non-zero contribution, so the sum is exact).

        combine == 'fit': the lists of the fitted combination (utils.recommend_combined), one top-N call per owner group
        with that group's T_g; on several GPUs the same placement by owner shard and the same exact all-reduce."""
        if self._use_fit():
            return self._recommend_combined(users, top_n, exclude)
        qsum = self._item_sum_in_shard_order()
        P = self.model_list[0].user_mat.weight.data
        u = _request_users(users, self.n_user, self.device)
        if self.dist.world == 1:
            return recommend_from_tables(P, qsum, self.n_group, u, top_n, exclude)
        owner = self._owner[u.long()]
        rank_of = torch.where(owner >= 0, owner % self.dist.world, torch.zeros_like(owner))
        pos = torch.nonzero(rank_of == self.dist.rank).flatten()
        items = torch.zeros((u.shape[0], top_n), dtype=torch.int32, device=self.device)
        scores = torch.zeros((u.shape[0], top_n), dtype=torch.float32, device=self.device)
        if pos.numel() > 0:
            it, sc = recommend_from_tables(P, qsum, self.n_group, u[pos], top_n, exclude)
            items[pos] = it
            scores[pos] = sc
        self.dist.all_reduce(items)
        self.dist.all_reduce(scores)
        return items, scores

    # ------------------------------------------------------------------ learned combination (combine == 'fit')
    def _use_fit(self):
        """True when the evaluation and recommend use the fitted combination; combine must be 'mean' or 'fit'."""
        if self.combine not in ('mean', 'fit'):
            raise ValueError(f"Sisa.combine must be 'mean' or 'fit', not {self.combine!r}")
        if self.combine == 'fit' and self.loss == 'bpr':
            raise ValueError("Sisa.combine='fit' cannot combine BPR shard models: the fit is least squares on the "
                             "ratings, and BPR scores are not ratings; use combine='mean'")
        return self.combine == 'fit'

    def _fitted(self):
        """The combination the last learn / unlearn pass fitted, or a clear error when it did not fit one."""
        if self.combination is None:
            raise RuntimeError("Sisa.combine == 'fit' but no combination has been fitted: run learn or unlearn with "
                               "combine='fit' first")
        return self.combination

    def _item_tables_in_shard_order(self):
        """[Q_0 .. Q_{K-1}] on this GPU.  On several GPUs the ranks all-gather their item tables chunk by chunk of item
        rows, as _item_sum_in_shard_order does, into one [K, n_item, d] buffer: every rank then holds the same bits."""
        K, world, rank = self.n_group, self.dist.world, self.dist.rank
        if world == 1:
            return [self.model_list[s].item_mat.weight.data for s in range(K)]
        slots = -(-K // world)
        rows = max(1, min(self.n_item, self.RECOMMEND_GATHER_BYTES // (world * slots * self.k * 4)))
        part = torch.zeros((slots, rows, self.k), dtype=torch.float32, device=self.device)
        full = torch.empty((world * slots, rows, self.k), dtype=torch.float32, device=self.device)
        Q = torch.empty((K, self.n_item, self.k), dtype=torch.float32, device=self.device)
        mine = list(range(rank, K, world))
        for r0 in range(0, self.n_item, rows):
            n = min(self.n_item, r0 + rows) - r0
            for j, s in enumerate(mine):
                part[j, :n].copy_(self.model_list[s].item_mat.weight.data[r0:r0 + n])
            self.dist.all_gather_into(full, part)
            for s in range(K):
                Q[s, r0:r0 + n].copy_(full[(s % world) * slots + s // world, :n])
        return list(Q)

    def _fit_combination(self, train_dlist, save_dir):
        """Fit the combination of every owner group on this pass's training rows (after an unlearn: the retained rows
        only) -- every group, because retrained shards change every group's features.  Every rank fits every group
        from the same gathered tables, so all ranks hold the same weights.  combine.npy: fp64 [K, K + 1], (w_g, b_g)."""
        recs = [train_dlist[g].dataset.records(self.device) for g in range(self.n_group)]
        self.combination = fit_combination(self.model_list[0].user_mat.weight.data, self._item_tables_in_shard_order(),
                                           recs)
        if len(save_dir) > 0 and self.dist.rank == 0:
            np.save(save_dir + '/combine', self.combination.table())

    def _combined_test(self, test_data, verbose):
        """The final evaluation under the fitted combination: ure_group_score, then ure_rank_metrics.  On several GPUs
        with the per-shard test sets partitioning test_data (as in _ensemble_test_sharded), every rank scores the test
        rows of the groups whose owner shard it holds and the sums are all-reduced; otherwise every rank evaluates the
        whole test set."""
        dev, K, c = self.device, self.n_group, self._fitted()
        P = self.model_list[0].user_mat.weight.data
        tdl = getattr(self, '_test_dlist', None)
        sharded = self.dist.world > 1 and self.eval_sharded is not False and tdl is not None and len(tdl) == K and \
            sum(len(t.dataset) for t in tdl) == len(test_data.dataset)
        out = torch.zeros(5, dtype=torch.float64, device=dev)
        if sharded:
            recs = [tdl[i].dataset.records(dev) for i in self.dist.my_shards(range(K)) if len(tdl[i].dataset) > 0]
            rows = _eval_rows(recs, self.n_user) if recs else None
        else:
            ds = test_data.dataset
            rows = (ds.records(dev),) + tuple(ds.segments(dev, self.n_user)) if len(ds) > 0 else None
        if rows is not None:
            inter, order, seg = rows
            score, _ = kn.group_score(P, c.T, c.b_slot, self._owner, inter, sse=out[0:1])
            kn.rank_metrics(inter, score, seg, order, out=out[1:4])
        if sharded:
            sb = getattr(self, '_last_batch', None)
            if sb is not None and getattr(sb, 'optimistic', False):
                out[4:5].copy_(sb.ws[16:20].view(torch.int32))     # as in _ensemble_test_sharded
            self.dist.all_reduce(out)
        vals = kn.download_many([out])[0]
        if vals[4] > 0:
            raise kn.PlanHintMiss("ultrare_b200: a rank's remembered owner plan did not cover its batch")
        rmse, ndcg, hr = base_test_values(vals[:4], len(test_data.dataset))
        if verbose == 2:
            print(f'Test - RMSE: {rmse:>.4f}, NDCG: {ndcg:>.3f}, HR: {hr:>.3f}')
        return rmse, ndcg, hr

    def _recommend_combined(self, users, top_n, exclude):
        P = self.model_list[0].user_mat.weight.data
        u = _request_users(users, self.n_user, self.device)
        if self.dist.world == 1:
            return recommend_combined(P, self._fitted(), self._owner, u, top_n, exclude)
        owner = self._owner[u.long()]
        keep = torch.where(owner >= 0, owner % self.dist.world, torch.zeros_like(owner)) == self.dist.rank
        items, scores = recommend_combined(P, self._fitted(), self._owner, u, top_n, exclude, keep=keep)
        self.dist.all_reduce(items)
        self.dist.all_reduce(scores)
        return items, scores

    def _ensemble_test_sharded(self, test_dlist):
        """Multi-GPU evaluation with the TEST ROWS sharded: every rank scores the test sets of its own shards (the
        rows of the users it owns) and the four sums are all-reduced; a rank uploads and segments only its own test
        rows.  Equal to evaluating the merged set because the per-shard test sets partition it by user
        (config.py:144-148).  After the merge every model shares ONE user table, so the ensemble mean
        (1/K) sum_k P[u].Q_k[i] is P[u].(sum_k Q_k[i]) / K: the ranks all-reduce the sum of their item tables
        ([n_item, d]) instead of n_test partial scores, and a test row costs one item gather instead of K."""
        dev, K = self.device, self.n_group
        mine = [i for i, m in enumerate(self.model_list) if getattr(m, 'item_mat', None) is not None]
        if mine:
            qs = [self.model_list[i].item_mat.weight.data for i in mine]
            block = _as_one_block(qs)      # the item tables of a batch arena: one reduction, no stack copy
            qsum = block.view(len(qs), self.n_item, self.k).sum(0) if block is not None else torch.stack(qs).sum(0)
        else:
            qsum = torch.zeros((self.n_item, self.k), dtype=torch.float32, device=dev)
        self.dist.all_reduce(qsum)
        merged = self.model_list[0].user_mat.weight.data
        out = torch.zeros(5, dtype=torch.float64, device=dev)
        recs = [test_dlist[i].dataset.records(dev) for i in mine if len(test_dlist[i].dataset) > 0]
        if recs:
            inter, order, seg = _eval_rows(recs, self.n_user)
            score, sse = kn.ensemble_score([merged], [qsum], inter, denom=float(K))
            out[0:1] = sse
            out[1:4] = kn.rank_metrics(inter, score, seg, order)
        sb = getattr(self, '_last_batch', None)
        if sb is not None and getattr(sb, 'optimistic', False):
            # this rank's error word (0, or 2 = the remembered plan was not covered), one converting copy
            out[4:5].copy_(sb.ws[16:20].view(torch.int32))
        self.dist.all_reduce(out)
        vals = kn.download_many([out])[0]
        if vals[4] > 0:                        # on some rank: every rank repeats the pass (Sisa._retrying)
            raise kn.PlanHintMiss("ultrare_b200: a rank's remembered owner plan did not cover its batch")
        n_test = sum(len(t.dataset) for t in test_dlist)
        users = max(vals[3], 1.0)
        return float(np.sqrt(vals[0] / max(1, n_test))), float(vals[1] / users), float(vals[2] / users)

    def _ensemble_test(self, test_data, verbose):
        if self.dist.world == 1:
            return baseTest(test_data, self.model_list, self.loss_fn, self.device, verbose)
        tdl = getattr(self, '_test_dlist', None)
        if self.eval_sharded is not False and tdl is not None and len(tdl) == self.n_group and \
                sum(len(t.dataset) for t in tdl) == len(test_data.dataset):
            return self._ensemble_test_sharded(tdl)
        # every rank scores against its own shards' item tables; partial sums are all-reduced
        mine = _local(self.model_list)
        ds = test_data.dataset
        inter = ds.records(self.device)
        if mine:
            part, _ = kn.ensemble_score([m.user_mat.weight.data for m in mine],
                                        [m.item_mat.weight.data for m in mine], inter, denom=1.0)
        else:
            part = torch.zeros(len(ds), dtype=torch.float32, device=self.device)
        self.dist.all_reduce(part)
        score, sse = kn.score_finalize(part, inter, float(self.n_group))
        # ranking metrics: every rank takes its block of the user segments, the three sums are all-reduced
        order, seg = ds.segments(self.device, self.n_user)
        lo, hi = self.dist.row_block(seg.shape[0] - 1)
        out = kn.rank_metrics(inter, score, seg[lo:hi + 1], order) if hi > lo else \
            torch.zeros(3, dtype=torch.float64, device=self.device)
        self.dist.all_reduce(out)
        vals = torch.cat([sse, out]).cpu().numpy()
        users = max(vals[3], 1.0)
        return float(np.sqrt(vals[0] / len(ds))), float(vals[1] / users), float(vals[2] / users)

    # ------------------------------------------------------------------ batched shard training
    def _train_shards(self, ids, train_dlist, test_dlist, test_data, verbose, prior, defer_logs=False):
        """Train shards `ids` (ascending) together; returns ({shard: model}, {shard: unmerged P},
        {shard: index of its last-epoch log entry}).

        prior(i, new) -> list of models the reference would have in self.model_list while shard
        i trains, `new` being the {shard: model} dict of this call (epoch_eval='faithful' only).
        """
        mine = self.dist.my_shards(list(ids))
        self._last_batch = None
        mode = self._mode()
        compact = mode != 'faithful'
        E = self.epochs
        t0 = time.time()
        models, states, snaps, losses = {}, [], {}, []
        if mine:
            # default init: the native batch runtime (kernels.ArenaShardBatch) -- ONE allocation, one library call
            # that queues the descriptor table, the clears and the owner set-up, one normal_() for every table of
            # the launch (device RNG); an overridden _new_model (parity runs inject weights), host-seeded init or
            # explicit visiting orders go shard by shard
            batched = self.init_on_device and type(self)._new_model is Scratch._new_model
            # the staging copies of the shards' records run on worker threads while the models are allocated
            from ..read import RatingData
            from .utils import MF
            uploaded = RatingData.upload_many([train_dlist[i].dataset for i in mine], self.device,
                                              self._row_of if compact else None, 'sisa_local' if compact else None,
                                              defer=True)
            t_a = time.time()
            uploaded()
            recs = [(train_dlist[i].dataset.records_mapped(self.device, self._row_of, 'sisa_local') if compact
                     else train_dlist[i].dataset.records(self.device)) for i in mine]
            batch = train_dlist[mine[0]].batch_size
            t_b = time.time()
            if batched:
                from .scratch import model_generator
                # optimistic launch (kernels.ArenaShardBatch): only when the losses are read after the evaluation;
                # several GPUs: only with the row-sharded final evaluation, whose all-reduce carries every rank's
                # "plan not covered" flag, so that all ranks repeat the pass together
                will_shard_eval = self.dist.world > 1 and self.eval_sharded is not False and test_data is not None and \
                    sum(len(t.dataset) for t in test_dlist) == len(test_data.dataset)
                optimistic = defer_logs and mode == 'none' and verbose != 1 and (self.dist.world == 1 or will_shard_eval)
                rows = [len(self.group_index[i]) if compact else self.n_user for i in mine]
                perms = [train_dlist[i].explicit_perm(self.device, E) for i in mine]
                sb = kn.ArenaShardBatch(recs, rows, self.n_item, self.k, batch, E, [i + 1 for i in mine], self.seed,
                                        perms if any(p is not None for p in perms) else None, self.lr, self.lr_decay,
                                        50, self.lam, self.momentum,
                                        generator=lambda: model_generator(self.seed, mine[0] + 1, self.device),
                                        optimistic=optimistic, loss=self.loss)
                states = None
            else:
                for j, i in enumerate(mine):
                    models[i] = self._new_model(i + 1, user_rows=self._rows(i)) if compact else self._new_model(i + 1)
                    P, Q = models[i].user_mat.weight.data, models[i].item_mat.weight.data
                    states.append(kn.ShardState(recs[j], P, Q, E, shard_id=i + 1, perm_seed=self.seed,
                                                perm=train_dlist[i].explicit_perm(self.device, E)))
                sb = kn.ShardBatch(states, self.k, batch, self.lr, self.lr_decay, 50, self.lam, self.momentum,
                                   loss=self.loss)
            self.timing['setup_alloc_ms'] = (t_a - t0) * 1e3
            self.timing['setup_upload_states_ms'] = (t_b - t_a) * 1e3
            self.timing['setup_batch_ms'] = (time.time() - t_b) * 1e3
            self.timing['batch_ctor_ms'] = getattr(sb, 'ctor_ms', None)
            if states is None and mode == 'faithful':
                states = sb.shards
            if mode == 'faithful':
                need = sum((s.P.numel() + s.Q.numel()) * 4 for s in states) * E
                if need > 8 << 30:
                    warnings.warn("epoch_eval='faithful' needs %.1f GB of snapshots; evaluating the last epoch only"
                                  % (need / 2**30))
                    mode = 'faithful-last'
            if mode == 'faithful':
                ends = {}
                for j, s in enumerate(states):
                    spe = s.steps_per_epoch(batch)
                    for e in range(E):
                        ends.setdefault((e + 1) * spe, []).append((j, e))
                for boundary in sorted(ends):
                    sb.train(boundary)
                    for j, e in ends[boundary]:
                        snaps[(mine[j], e)] = (states[j].P.clone(), states[j].Q.clone())
            else:
                self.timing['setup_ms'] = (time.time() - t0) * 1e3
                sb.train()
                self.timing['launch_ms'] = (time.time() - t0) * 1e3 - self.timing['setup_ms']
                if batched:
                    states = sb.shards                                  # the per-shard views, while the GPU trains
                    for j, i in enumerate(mine):
                        models[i] = MF.wrap(states[j].P, states[j].Q)
                # while the GPU trains: the model wrappers, and what the final evaluation needs (upload + user
                # segments are cached on the RatingData objects), so self.test() after the merge finds them resident
                sharded_eval = self.dist.world > 1 and self.eval_sharded is not False and test_data is not None and \
                    sum(len(t.dataset) for t in test_dlist) == len(test_data.dataset)
                # ... on a side stream: queued behind the training launch on the SAME stream the uploads would wait
                # for the training kernel to end (measured: 70 us of H2D + pack on the critical path after it); the
                # copy engine is free while the SMs train.  The main stream waits for the side stream before the merge.
                main = torch.cuda.current_stream(self.device)
                side = kn.side_stream(self.device)
                with torch.cuda.stream(side):
                    fresh = []
                    if sharded_eval:                # the final evaluation reads this rank's own test rows only
                        for i in mine:
                            if len(test_dlist[i].dataset) > 0:
                                fresh.append(test_dlist[i].dataset.records(self.device))
                    for ld in ([test_data] if test_data is not None and not sharded_eval else []) + \
                            ([test_dlist[i] for i in mine] if mode == 'final' and self.dist.world == 1 else []):
                        ds = getattr(ld, 'dataset', None)
                        if ds is not None and len(ds) > 0:
                            fresh.append(ds.records(self.device))
                            fresh.extend(t for t in ds.segments(self.device, self.n_user) if t is not None)
                    for t in fresh:
                        t.record_stream(main)
                main.wait_stream(side)
            if batched and not models:
                states = sb.shards
                for j, i in enumerate(mine):
                    models[i] = MF.wrap(states[j].P, states[j].Q)
            self._last_batch = sb
            # defer_logs: the loss read-back is queued and awaited after the final evaluation (_flush_logs), so
            # the merge and the evaluation are launched while the GPU still trains
            defer_logs = defer_logs and mode == 'none' and verbose != 1
            pending = sb.train_losses_async()
            losses = None if defer_logs else pending()       # the one sync of the whole training
        else:
            defer_logs = False
        self.timing['train_s'] = time.time() - t0
        unmerged = {i: models[i].user_mat.weight.data for i in mine}
        if defer_logs:
            self._pending_logs = lambda: self._write_logs(mine, pending(), mode, models, states, snaps, prior,
                                                          test_dlist, test_data, verbose)
            return models, unmerged, {}, compact
        last_idx = self._write_logs(mine, losses, mode, models, states, snaps, prior, test_dlist, test_data, verbose)
        return models, unmerged, last_idx, compact

    def _flush_logs(self):
        """Write the training-log entries whose loss read-back was deferred (after the evaluation's sync)."""
        pend, self._pending_logs = getattr(self, '_pending_logs', None), None
        if pend is not None:
            pend()

    def _write_logs(self, mine, losses, mode, models, states, snaps, prior, test_dlist, test_data, verbose):
        E = self.epochs

        # ---- logs, in the reference's order: shard after shard, epoch after epoch (Appendix A14)
        nan = float('nan')
        last_idx = {}
        stamp = time.strftime('%H:%M:%S', time.gmtime(self.timing['train_s'] / max(1, E * max(1, len(mine)))))
        if not mode.startswith('faithful') and verbose != 1:
            # no per-epoch evaluation and nothing to print: whole columns at once
            for j, i in enumerate(mine):
                self.log['train_loss'].extend(np.asarray(losses[j], dtype=np.float64).tolist())
                for key in ('test_rmse', 'test_ndcg', 'test_hr', 'total_rmse', 'total_ndcg', 'total_hr'):
                    self.log[key].extend([nan] * E)
                self.log['time'].extend([stamp] * E)
                last_idx[i] = len(self.log['test_rmse']) - 1
            return last_idx
        # per-epoch evaluations (scratch.py:83-97): ALL of them are queued first -- two launches each, no
        # synchronisation -- and their sums come back in one transfer (round 1 synchronised after every baseTest:
        # 2 x epochs x shards host round trips)
        # ... as JOBS of one pair of launches (ure_eval_jobs, grid.y = job): two baseTest calls per shard and epoch
        # were 4 launches each, 2000 launches for K = 5, E = 50 -- the default mode was launch-bound at ~90 ms per pass
        keys, jobs, sizes = [], [], []
        dev = self.device
        for j, i in enumerate(mine):
            pri = prior(i, models) if mode.startswith('faithful') else None
            for e in range(E):
                if mode == 'faithful' or (mode == 'faithful-last' and e == E - 1):
                    P, Q = snaps[(i, e)] if mode == 'faithful' else (states[j].P, states[j].Q)
                    Ps = [m.user_mat.weight.data for m in pri] + [P]
                    Qs = [m.item_mat.weight.data for m in pri] + [Q]
                    keys.append((i, e))
                    for ld in (test_dlist[i], test_data):
                        ds = ld.dataset
                        order, seg = ds.segments(dev, Ps[0].shape[0])
                        jobs.append((Ps, Qs, ds.records(dev), order, seg))
                        sizes.append(len(ds))
        results = {}
        chunk = max(2, int((1 << 30) // (4 * max([1] + sizes))) // 2 * 2)        # <= 1 GB of score scratch per launch
        for c0 in range(0, len(jobs), chunk):
            live = [x for x in range(c0, min(len(jobs), c0 + chunk)) if sizes[x] > 0]
            vals = kn.download_many([kn.eval_jobs([jobs[x] for x in live], self.k)])[0] if live else np.zeros((0, 4))
            got = {x: vals[y] for y, x in enumerate(live)}
            for x in range(c0, min(len(jobs), c0 + chunk), 2):
                results[keys[x // 2]] = tuple(base_test_values(got.get(x + w, np.zeros(4)), sizes[x + w]) for w in (0, 1))
        for j, i in enumerate(mine):
            for e in range(E):
                self.log['train_loss'].append(float(losses[j][e]))
                tr, to = results.get((i, e), ((nan, nan, nan), (nan, nan, nan)))
                for key, v in zip(('test_rmse', 'test_ndcg', 'test_hr'), tr):
                    self.log[key].append(v)
                for key, v in zip(('total_rmse', 'total_ndcg', 'total_hr'), to):
                    self.log[key].append(v)
                self.log['time'].append(stamp)
                if verbose == 1:
                    print(f'[shard {i+1}] Epoch: [{e+1:>2d}/{E:>2d}] train loss: {losses[j][e]:>.9f},'
                          f' test RMSE: {tr[0]:>.4f}, total RMSE: {to[0]:>.4f}')
            last_idx[i] = len(self.log['test_rmse']) - 1
        return last_idx

    def _finish(self, new, unmerged, last_idx, compact, merged, test_dlist, save_dir):
        """After the merge: 'final'-mode last-epoch test metrics, then the per-shard artefacts."""
        full_merged = nn.Parameter(merged, requires_grad=False)
        for i, m in new.items():
            m.user_mat = nn.Embedding(merged.shape[0], self.k, _weight=merged)
            m.user_mat.weight = full_merged
        if self._mode() == 'final' and self.dist.world == 1:
            # own shard's test users are all owned by shard i: merged rows == its rows.  One pair of launches and one
            # read-back for all shards (ure_eval_jobs) instead of four launches and a synchronisation per shard
            ids = [i for i in new if len(test_dlist[i].dataset) > 0]
            jobs = []
            for i in ids:
                ds = test_dlist[i].dataset
                order, seg = ds.segments(self.device, merged.shape[0])
                jobs.append(([new[i].user_mat.weight.data], [new[i].item_mat.weight.data], ds.records(self.device), order, seg))
            vals = kn.download_many([kn.eval_jobs(jobs, self.k)])[0] if jobs else []
            for i in new:
                tr = base_test_values(vals[ids.index(i)], len(test_dlist[i].dataset)) if i in ids else (0.0, 0.0, 0.0)
                for key, v in zip(('test_rmse', 'test_ndcg', 'test_hr'), tr):
                    self.log[key][last_idx[i]] = v
        if len(save_dir) > 0 and new:
            # artefacts (scratch.py:131-144 per shard): ONE pinned device-to-host transfer for all tables, the
            # files are written by a worker thread while the final evaluation runs (_join_writers waits for them)
            tensors = []
            for i, m in new.items():
                P = unmerged[i]
                if compact:                # artefact keeps the reference's [n_user, k] shape; non-owner rows zero
                    full = torch.zeros((self.n_user, self.k), dtype=torch.float32, device=self.device)
                    full[self._rows(i)] = P
                    P = full
                tensors += [P, m.item_mat.weight.data]
            host = kn.download_many(tensors)
            log = {k: list(v) for k, v in self.log.items()}

            # log{i}.npy is written by the reference as shard i finishes (scratch.py:144): it holds the entries
            # accumulated up to and including shard i's last epoch, not the whole run's log
            cut = {i: last_idx.get(i, len(log['train_loss']) - 1) + 1 for i in new}

            def write(ids=list(new), host=host, log=log, cut=cut):
                for j, i in enumerate(ids):
                    P_h, Q_h = host[2 * j], host[2 * j + 1]
                    torch.save({'user_mat.weight': torch.from_numpy(P_h), 'item_mat.weight': torch.from_numpy(Q_h)},
                               save_dir + '/model' + str(i + 1) + '.pth')
                    np.save(save_dir + '/user_mat' + str(i + 1), P_h)
                    np.save(save_dir + '/item_mat' + str(i + 1), Q_h)
                    np.save(save_dir + '/log' + str(i + 1), {k: v[:cut[i]] for k, v in log.items()})

            self._writers.append(_writer_pool().submit(write))

    def _join_writers(self):
        """Wait for the artefact files of this learn / unlearn call (raises what a writer raised)."""
        pending, self._writers = self._writers, []
        for f in pending:
            f.result()

    # ------------------------------------------------------------------ merge
    def _merged_from(self, base, unmerged, compact, retrain_flags):
        """Owner rows of the freshly trained shards gathered over `base` (or zeros): sisa.py:52-58,107-113."""
        dev, K = self.device, self.n_group
        filler = next(iter(unmerged.values())) if unmerged else base
        tables = [unmerged.get(s, filler) for s in range(K)]
        row_of = self._row_of if compact else None
        if self.dist.world == 1:
            merged = torch.zeros((self.n_user, self.k), dtype=torch.float32, device=dev) if base is None else base.clone()
            kn.merge_user_rows(tables, self._owner, merged, row_of=row_of, retrain=retrain_flags,
                               zero_unowned=base is None)
            return merged
        # multi-GPU: each rank contributes the rows of the shards it trained.  Owner rows are disjoint, so the ranks
        # ALL-GATHER their compact tables (each rank's shards back to back, padded to the longest rank) -- every
        # row crosses NVLink once -- and the merge kernel gathers from the gathered buffer through per-shard base
        # pointers.  (Round 1 all-reduced a zero-filled [n_user, k] table: twice the bytes.)
        t0 = time.perf_counter()
        trained = sorted(self.retrain_gid) if base is not None else list(range(K))
        sizes = {s_: (len(self.group_index[s_]) if compact else self.n_user) for s_ in trained}
        by_rank = {}
        for s_ in trained:
            by_rank.setdefault(self.dist.owner_of_shard(s_), []).append(s_)
        maxlen = max([sum(sizes[s_] for s_ in v) for v in by_rank.values()] or [1])
        mine_now = by_rank.get(self.dist.rank, [])
        block = _as_one_block([unmerged[s_] for s_ in mine_now])
        if block is not None and block.shape[0] == maxlen:
            send = block                   # this rank's owner rows are one run of the batch arena: gathered in place
        else:
            send = torch.empty((maxlen, self.k), dtype=torch.float32, device=dev)
            o = 0
            for s_ in mine_now:
                send[o:o + sizes[s_]].copy_(unmerged[s_], non_blocking=True)
                o += sizes[s_]
        gathered = torch.empty((self.dist.world * maxlen, self.k), dtype=torch.float32, device=dev)
        t1 = time.perf_counter()
        self.dist.all_gather_into(gathered, send)
        self.timing['merge_local_ms'] = (t1 - t0) * 1e3
        self.timing['merge_allgather_ms'] = (time.perf_counter() - t1) * 1e3
        tables, flags_np = [gathered] * K, np.zeros(K, dtype=np.int32)
        for r_, v in by_rank.items():
            o = r_ * maxlen
            for s_ in v:
                tables[s_] = gathered[o:o + sizes[s_]]
                flags_np[s_] = 1
                o += sizes[s_]
        merged = torch.zeros((self.n_user, self.k), dtype=torch.float32, device=dev) if base is None else base.clone()
        kn.merge_user_rows(tables, self._owner, merged, row_of=row_of, retrain=kn.upload_array(flags_np, dev),
                           zero_unowned=base is None)
        return merged

    # ------------------------------------------------------------------ learn / unlearn
    def _retrying(self, once, *args):
        """An optimistic owner launch whose remembered plan did not cover the batch trained nothing (kernels.PlanHintMiss,
        raised when the deferred losses are read): repeat the pass -- the hint is gone, so this one waits for its plan."""
        try:
            return once(*args)
        except kn.PlanHintMiss:
            kn._PLAN_HINTS.clear()
            self._pending_logs = None
            self._join_writers()
            return once(*args)

    def learn(self, train_dlist, test_dlist, test_data, verbose, save_dir):
        """reference sisa.py:25-63."""
        self._use_fit()                     # refuse a combine / loss conflict before anything trains
        if self._sliced():
            return self._learn_sliced(train_dlist, test_dlist, test_data, verbose, save_dir)
        return self._retrying(self._learn_once, train_dlist, test_dlist, test_data, verbose, save_dir)

    def _learn_once(self, train_dlist, test_dlist, test_data, verbose, save_dir):
        assert len(train_dlist) == self.n_group
        assert len(test_dlist) == self.n_group
        self._test_dlist = test_dlist
        new, unmerged, last_idx, compact = self._train_shards(
            range(self.n_group), train_dlist, test_dlist, test_data, verbose,
            lambda i, new: [new[j] for j in range(i)], defer_logs=len(save_dir) == 0)
        merged = self._merged_from(None, unmerged, compact, None)
        self._finish(new, unmerged, last_idx, compact, merged, test_dlist, save_dir)
        shared = next(iter(new.values())).user_mat.weight if new else nn.Parameter(merged, requires_grad=False)
        self.model_list = [new[i] if i in new else _RemoteModel(shared) for i in range(self.n_group)]
        if self._use_fit():
            t_c = time.perf_counter()
            self._fit_combination(train_dlist, save_dir)
            self.timing['combine_fit_ms'] = (time.perf_counter() - t_c) * 1e3
        self.test(test_data, verbose, save_dir)
        self._flush_logs()
        self._join_writers()
        return self.model_list

    ROUTE_ON_HOST_MAX = 1 << 14     # deletion sets up to this size are routed from the host copy of the owner map

    def route(self, del_user, defer_upload=False):
        """retrain flags of sisa.py:76-81 (int32 [n_group] on the device): flags[owner[u]] = 1 for every deleted u.
        Large deletion sets go through the owner-map kernel (ure_route_deletions); a small one is a few hundred
        look-ups in the host copy of the same owner map -- no device round trip before the shards can be set up
        (defer_upload: not even the upload of the flags; the caller sends them when the merge needs them)."""
        ids = np.asarray(list(del_user), dtype=np.int64)
        if self.slices > 1:
            self.first_slice = self._first_slices(ids)
        if len(ids) <= self.ROUTE_ON_HOST_MAX:
            own = self._owner_np[ids[(ids >= 0) & (ids < self.n_user)]]
            flags_h = np.zeros(self.n_group, dtype=np.int32)
            flags_h[own[own >= 0]] = 1
            self._route_flags_host = flags_h
            return None if defer_upload else kn.upload_array(flags_h, self.device)
        self._route_flags_host = None
        d = kn.upload_array(ids.astype(np.int32), self.device)
        return kn.route_deletions(self._owner, d, self.n_group)

    def _first_slices(self, ids):
        """int32 [n_group]: per shard the first slice holding a routed user, min over u of row_of[u] * R // m_g
        (R: no routed user), from the host copies of the owner and row maps."""
        R = self.slices
        ids = ids[(ids >= 0) & (ids < self.n_user)]
        own = self._owner_np[ids]
        ids, own = ids[own >= 0], own[own >= 0]
        sizes = np.array([max(1, len(g)) for g in self.group_index], dtype=np.int64)
        first = np.full(self.n_group, R, dtype=np.int32)
        np.minimum.at(first, own, (self._row_of_np[ids].astype(np.int64) * R // sizes[own]).astype(np.int32))
        return first

    def unlearn(self, model_list, train_dlist, test_dlist, test_data, del_user, verbose, save_dir):
        """reference sisa.py:66-118."""
        self._use_fit()
        if self._sliced():
            return self._unlearn_sliced(model_list, train_dlist, test_dlist, test_data, del_user, verbose, save_dir)
        return self._retrying(self._unlearn_once, model_list, train_dlist, test_dlist, test_data, del_user, verbose,
                              save_dir)

    def _unlearn_once(self, model_list, train_dlist, test_dlist, test_data, del_user, verbose, save_dir):
        self.model_list = list(model_list)
        assert len(train_dlist) == self.n_group
        assert len(test_dlist) == self.n_group

        self._test_dlist = test_dlist
        t_begin = time.perf_counter()
        flags = self.route(del_user, defer_upload=True)
        flags_h = self._route_flags_host if self._route_flags_host is not None else kn.download_many([flags])[0]
        self.retrain_gid = set(int(s) for s in np.flatnonzero(flags_h))
        self.timing['route_ms'] = (time.perf_counter() - t_begin) * 1e3
        order = sorted(self.retrain_gid)
        model_before_unlearn = self.model_list[0]                               # sisa.py:84
        base = model_before_unlearn.user_mat.weight.data
        old = list(self.model_list)

        def prior(i, new):
            # self.model_list as the reference sees it while retraining shard i: the old models, with
            # the shards retrained before i (ascending set order) already replaced (sisa.py:86-89)
            cur = [(new[j] if (j in new and j in order and order.index(j) < order.index(i)) else old[j])
                   for j in range(self.n_group)]
            return _local(cur)

        new, unmerged, last_idx, compact = self._train_shards(order, train_dlist, test_dlist, test_data, verbose, prior,
                                                              defer_logs=len(save_dir) == 0)
        t_m = time.perf_counter()
        if flags is None:                              # routed on the host: the flags go up while the GPU trains
            flags = kn.upload_array(self._route_flags_host, self.device, side=True)
        merged = self._merged_from(base, unmerged, compact, flags)
        self._finish(new, unmerged, last_idx, compact, merged, test_dlist, save_dir)
        for i, m in new.items():
            self.model_list[i] = m
        shared = next(iter(new.values())).user_mat.weight if new else nn.Parameter(merged, requires_grad=False)
        for m in self.model_list:
            m.user_mat.weight = shared
        t_c = time.perf_counter()
        fit = self._use_fit()
        if fit:
            self._fit_combination(train_dlist, save_dir)
            self.timing['combine_fit_ms'] = (time.perf_counter() - t_c) * 1e3
        t_t = time.perf_counter()
        self.test(test_data, verbose, save_dir)
        self.timing['merge_ms'] = (t_c - t_m) * 1e3
        # kernels of ours outside the training batch: route (large deletion sets only), merge, score, ranking; with the
        # fitted combination also the Gram, its fold and the weighted item sum
        self.timing['own_launches_outside_batch'] = (0 if self._route_flags_host is not None else 1) + 1 + 2 + \
            (3 if fit else 0)
        self._flush_logs()
        self._join_writers()
        self.timing['test_ms'] = (time.perf_counter() - t_t) * 1e3
        self.timing['total_ms'] = (time.perf_counter() - t_begin) * 1e3
        return self.model_list

    # ------------------------------------------------------------------ SISA slicing (slices > 1)
    def _sliced(self):
        """True when learn / unlearn train in slice stages; checks what slicing needs."""
        R = self.slices
        if not isinstance(R, (int, np.integer)) or not 1 <= R <= 32:
            raise ValueError(f"Sisa.slices must be an integer in 1..32, not {R!r}")
        if R == 1:
            return False
        if self.epoch_eval not in ('final', 'none'):
            raise ValueError(f"Sisa.slices > 1 needs epoch_eval 'final' or 'none', not {self.epoch_eval!r}")
        if not self.init_on_device or type(self)._new_model is not Scratch._new_model:
            raise ValueError("Sisa.slices > 1 needs the device-side initialisation of the batched shard training")
        return True

    def _slice_offsets(self, ds, g):
        """int64 [R + 1]: the slice boundaries of shard g's records, which must be slice-major (read with
        n_slice=R): the partition's offsets when the device ingest produced them, else counted from the users."""
        R = self.slices
        off = getattr(ds, 'slice_off', None)
        if off is None:
            s = self._row_of_np[np.asarray(ds.users, dtype=np.int64)].astype(np.int64) * R // \
                max(1, len(self.group_index[g]))
            if len(s) > 1 and (np.diff(s) < 0).any():
                raise ValueError(f"shard {g}: the training records are not slice-major; read them with n_slice={R}")
            off = np.concatenate([[0], np.cumsum(np.bincount(s, minlength=R))])
        off = np.asarray(off, dtype=np.int64)
        if off.shape != (R + 1,) or off[-1] != len(ds):
            raise ValueError(f"shard {g}: slice offsets {off.tolist()} do not describe {len(ds)} records in {R} slices")
        return off

    def _train_sliced(self, ids, first, ckpts, train_dlist, verbose, fresh):
        """Round j = 1..R trains stage j of every shard of `ids` on this GPU with first[g] < j, in one batch launch:
        E' epochs on the shard's slices 0..j-1, from the checkpoint ckpts[g][j-1] (fresh: round 1 draws the initial
        weights as the unsliced learn does, and they become checkpoint 0).  Returns ({shard: model}, {shard:
        unmerged P}, {shard: index of its last log entry}); every model carries its R checkpoints."""
        from ..read import RatingData
        from .scratch import model_generator
        from .utils import MF
        R, E1, dev = self.slices, stage_epochs(self.epochs, self.slices), self.device
        mine = self.dist.my_shards(list(ids))
        self._last_batch = None
        t0 = time.time()
        RatingData.upload_many([train_dlist[g].dataset for g in mine], dev, self._row_of, 'sisa_local')
        recs, offs, ck = {}, {}, {}
        for g in mine:
            if train_dlist[g].explicit_perm(dev, E1) is not None:
                raise ValueError(f"shard {g}: slice stages visit the keyed shuffled order; explicit orders are not "
                                 "supported with Sisa.slices > 1")
            recs[g] = train_dlist[g].dataset.records_mapped(dev, self._row_of, 'sisa_local')
            offs[g] = self._slice_offsets(train_dlist[g].dataset, g)
            ck[g] = list(ckpts[g])
        batch = train_dlist[mine[0]].batch_size if mine else self.batch
        models, pending, rounds, trained = {}, [], 0, 0
        for j in range(1, R + 1):
            due = [g for g in mine if first[g] < j]
            if not due:
                continue
            draw = fresh and j == 1
            # sliced rounds wait for their owner plan (no optimistic launch): PlanHintMiss cannot arise mid-pass
            sb = kn.ArenaShardBatch([recs[g][:int(offs[g][j])] for g in due], [len(self.group_index[g]) for g in due],
                                    self.n_item, self.k, batch, E1, [g + 1 for g in due], self.seed, None, self.lr,
                                    self.lr_decay, 50, self.lam, self.momentum,
                                    generator=lambda: model_generator(self.seed, mine[0] + 1, dev),
                                    init=None if draw else [ck[g][j - 1] for g in due], loss=self.loss)
            views = sb.shards
            if draw:
                for v, g in zip(views, due):
                    ck[g][0] = (v.P.clone(), v.Q.clone())
            sb.train()
            for v, g in zip(views, due):
                if j < R:
                    ck[g][j] = (v.P.clone(), v.Q.clone())
                else:
                    models[g] = MF.wrap(v.P, v.Q)
                    models[g].checkpoints = ck[g]
            pending.append((due, j, sb.train_losses_async()))
            rounds += 1
            trained += sb.interactions_trained()
        stages = {g: [] for g in mine}
        for due, j, wait in pending:
            for g, l in zip(due, wait()):
                stages[g].append((j, l))
        self.timing['train_s'] = time.time() - t0
        self.timing['rounds'] = rounds
        self.timing['trained_interactions'] = trained
        self.timing['stage_epochs'] = E1
        # logs: shard after shard, stage after stage, one train_loss entry per trained epoch (test_* NaN; 'final'
        # fills each shard's last entry in _finish)
        nan, last_idx = float('nan'), {}
        n_ep = sum(len(v) for v in stages.values()) * E1
        stamp = time.strftime('%H:%M:%S', time.gmtime(self.timing['train_s'] / max(1, n_ep)))
        for g in mine:
            for j, l in stages[g]:
                for e, v in enumerate(np.asarray(l, dtype=np.float64).tolist()):
                    self.log['train_loss'].append(v)
                    for key in ('test_rmse', 'test_ndcg', 'test_hr', 'total_rmse', 'total_ndcg', 'total_hr'):
                        self.log[key].append(nan)
                    self.log['time'].append(stamp)
                    if verbose == 1:
                        print(f'[shard {g+1}] Stage: [{j}/{R}] Epoch: [{e+1:>2d}/{E1:>2d}] train loss: {v:>.9f}')
            last_idx[g] = len(self.log['train_loss']) - 1
        return models, {g: models[g].user_mat.weight.data for g in mine}, last_idx

    def _learn_sliced(self, train_dlist, test_dlist, test_data, verbose, save_dir):
        assert len(train_dlist) == self.n_group
        assert len(test_dlist) == self.n_group
        self._test_dlist = test_dlist
        K, R = self.n_group, self.slices
        new, unmerged, last_idx = self._train_sliced(range(K), [0] * K, {g: [None] * R for g in range(K)},
                                                     train_dlist, verbose, fresh=True)
        merged = self._merged_from(None, unmerged, True, None)
        self._finish(new, unmerged, last_idx, True, merged, test_dlist, save_dir)
        shared = next(iter(new.values())).user_mat.weight if new else nn.Parameter(merged, requires_grad=False)
        self.model_list = [new[i] if i in new else _RemoteModel(shared) for i in range(K)]
        if self._use_fit():
            t_c = time.perf_counter()
            self._fit_combination(train_dlist, save_dir)
            self.timing['combine_fit_ms'] = (time.perf_counter() - t_c) * 1e3
        self.test(test_data, verbose, save_dir)
        self._join_writers()
        return self.model_list

    def _unlearn_sliced(self, model_list, train_dlist, test_dlist, test_data, del_user, verbose, save_dir):
        """Every shard with a routed user retrains from the checkpoint before its first affected slice a[g], on the
        retained records, stages a[g]+1 .. R; its checkpoints from a[g]+1 on are replaced.  Equal to a sliced learn
        on the retained data: no checkpoint it resumes from saw a deleted record."""
        self.model_list = list(model_list)
        assert len(train_dlist) == self.n_group
        assert len(test_dlist) == self.n_group
        self._test_dlist = test_dlist
        R = self.slices
        t_begin = time.perf_counter()
        flags = self.route(del_user, defer_upload=True)
        first = self.first_slice
        self.retrain_gid = set(int(s) for s in np.flatnonzero(first < R))
        self.timing['route_ms'] = (time.perf_counter() - t_begin) * 1e3
        order = sorted(self.retrain_gid)
        ckpts = {}
        for g in self.dist.my_shards(order):
            c = getattr(self.model_list[g], 'checkpoints', None)
            if c is None or len(c) != R:
                have = 'none' if c is None else f'{len(c)} slices'
                raise RuntimeError(f"Sisa.unlearn with slices={R}: shard {g}'s model holds no checkpoints for {R} "
                                   f"slices ({have}); learn with the same Sisa.slices first")
            ckpts[g] = c
        base = self.model_list[0].user_mat.weight.data
        new, unmerged, last_idx = self._train_sliced(order, first, ckpts, train_dlist, verbose, fresh=False)
        if flags is None:
            flags = kn.upload_array(self._route_flags_host, self.device, side=True)
        merged = self._merged_from(base, unmerged, True, flags)
        self._finish(new, unmerged, last_idx, True, merged, test_dlist, save_dir)
        for i, m in new.items():
            self.model_list[i] = m
        shared = next(iter(new.values())).user_mat.weight if new else nn.Parameter(merged, requires_grad=False)
        for m in self.model_list:
            m.user_mat.weight = shared
        if self._use_fit():
            t_c = time.perf_counter()
            self._fit_combination(train_dlist, save_dir)
            self.timing['combine_fit_ms'] = (time.perf_counter() - t_c) * 1e3
        self.test(test_data, verbose, save_dir)
        self._join_writers()
        self.timing['total_ms'] = (time.perf_counter() - t_begin) * 1e3
        return self.model_list

    # ------------------------------------------------------------------ state on disk and deletion requests
    def save_state(self, state_dir):
        """Write the model as a state directory (DESIGN.md §4.10): this rank's shards' item tables and checkpoints; on
        rank 0 the merged user table, the grouping, the ledger, the fitted combination and -- after every rank's
        files, last -- manifest.json.  One device-to-host transfer per rank; the files are written by the artefact
        writer thread.  A directory that already holds a manifest is refused: states are never overwritten."""
        from . import sisa_state as st
        src = self.source
        if src is None:
            raise ValueError("Sisa.save_state needs Sisa.source: the training data the model was learned from")
        if os.path.exists(os.path.join(state_dir, st.MANIFEST)):
            raise FileExistsError(f"{state_dir} already holds a SISA state; states are never overwritten")
        if len(self.model_list) != self.n_group:
            raise RuntimeError("Sisa.save_state: no trained model (run learn, or load a state, first)")
        K, R, rank = self.n_group, self.slices, self.dist.rank
        os.makedirs(state_dir, exist_ok=True)
        names, tensors = [], []
        for g in self.dist.my_shards(range(K)):
            m = self.model_list[g]
            names.append(f'item{g}')
            tensors.append(m.item_mat.weight.data)
            if R > 1:
                ck = getattr(m, 'checkpoints', None)
                if ck is None or len(ck) != R:
                    raise RuntimeError(f"Sisa.save_state with slices={R}: shard {g}'s model holds no {R} checkpoints")
                for r, (P, Q) in enumerate(ck):
                    names += [f'ckpt{g}_{r}_P', f'ckpt{g}_{r}_Q']
                    tensors += [P, Q]
        if rank == 0:
            names.append('merged')
            tensors.append(self.model_list[0].user_mat.weight.data)
        arrays = dict(zip(names, kn.download_many(tensors, copy=False)))
        if rank == 0:
            arrays['group_index_ids'], arrays['group_index_off'] = st.flat_index(src['group_index'])
            arrays['train_index_ids'], arrays['train_index_off'] = st.flat_index(self.group_index)
            arrays['deleted_users'] = np.asarray(self.deleted_users, dtype=np.int64)
            arrays['deleted_pairs'] = np.asarray(self.deleted_pairs, dtype=np.int64).reshape(-1, 2)
            if self._use_fit():
                arrays['combine'] = self._fitted().table()
                arrays['combine_gram'] = np.asarray(self._fitted().gram, dtype=np.float64)

        def write(arrays=arrays):
            for name, a in arrays.items():
                np.save(os.path.join(state_dir, name + '.npy'), a, allow_pickle=False)

        self._writers.append(_writer_pool().submit(write))
        self._join_writers()
        self.dist.barrier()                                     # every rank's files are on disk
        if rank == 0:
            if 'train_sha256' not in src:
                src['train_bytes'], src['train_sha256'] = st.file_digest(src['train_file'])
            man = dict(format=st.FORMAT_VERSION, K=K, slices=R, k=self.k, n_user=self.n_user, n_item=self.n_item,
                       epochs=self.epochs, batch=self.batch, lr=self.lr, lr_decay=self.lr_decay, lam=self.lam,
                       momentum=self.momentum, seed=self.seed, combine=self.combine, epoch_eval=self.epoch_eval,
                       loss=self.loss,
                       dataset=src['dataset'], grouping=src['grouping'], max_rating=src['max_rating'],
                       train_file=dict(path=os.path.abspath(src['train_file']), bytes=int(src['train_bytes']),
                                       sha256=src['train_sha256']),
                       test_file=os.path.abspath(src['test_file']), requests=int(self.requests),
                       saved_world_size=self.dist.world)
            path = os.path.join(state_dir, st.MANIFEST)
            with open(path + '.tmp', 'w') as f:
                json.dump(man, f, indent=1)
            os.replace(path + '.tmp', path)
        self.dist.barrier()

    @classmethod
    def load_state(cls, state_dir, param=None, dist=None):
        """The Sisa a state directory describes, ready for test / recommend / unlearn / apply_request: one MF per shard
        this rank holds (dist.my_shards, whatever the world size the state was saved at) sharing the merged user
        table, with its checkpoints when slices > 1; _RemoteModel for the other shards; the fitted combination
        rebuilt (ure_item_wsum) when combine == 'fit'.  ValueError for an incomplete state, another format version,
        a changed training file, or a `param` whose hyper-parameters differ from the state's."""
        from . import sisa_state as st
        from .utils import MF, combination_from
        man = st.read_manifest(state_dir)
        st.check_training_file(man)
        hp = types.SimpleNamespace(**{k: man[k] for k in ('n_user', 'n_item', 'k', 'lam', 'seed', 'lr', 'lr_decay',
                                                           'momentum', 'epochs', 'batch', 'loss')})
        for k, v in vars(hp).items():
            if param is not None and hasattr(param, k) and getattr(param, k) != v:
                raise ValueError(f"param.{k} = {getattr(param, k)!r}, but the state in {state_dir} has {k} = {v!r}")
        K, R = int(man['K']), int(man['slices'])
        group_index = st.unflat_index(st.load_array(state_dir, 'group_index_ids'),
                                      st.load_array(state_dir, 'group_index_off'))
        train_index = st.unflat_index(st.load_array(state_dir, 'train_index_ids'),
                                      st.load_array(state_dir, 'train_index_off'))
        if len(train_index) != K:
            raise ValueError(f"{state_dir}: train_index has {len(train_index)} groups, the manifest K = {K}")
        s = cls(hp, 'mf', K, train_index)
        if dist is not None:
            s.dist = dist
        s.epoch_eval, s.slices, s.combine = man['epoch_eval'], R, man['combine']
        s.source = dict(dataset=man['dataset'], train_file=man['train_file']['path'], test_file=man['test_file'],
                        max_rating=man['max_rating'], grouping=man['grouping'], group_index=group_index,
                        train_bytes=man['train_file']['bytes'], train_sha256=man['train_file']['sha256'])
        s.deleted_users = st.load_array(state_dir, 'deleted_users').astype(np.int64)
        s.deleted_pairs = st.load_array(state_dir, 'deleted_pairs').astype(np.int64).reshape(-1, 2)
        s.requests = int(man['requests'])

        def table(name, shape):
            a = st.load_array(state_dir, name)
            if a.dtype != np.float32 or a.shape != shape:
                raise ValueError(f"{state_dir}/{name}.npy is {a.dtype} {a.shape}, expected float32 {shape}")
            return a

        dev, d = s.device, s.k
        merged = kn.upload_table(table('merged', (s.n_user, d)), dev)
        shared = nn.Parameter(merged, requires_grad=False)
        mine = s.dist.my_shards(range(K))
        # this rank's item tables back to back in ONE allocation, as a learn's batch arena holds them
        Q = kn.upload_table(np.stack([table(f'item{g}', (s.n_item, d)) for g in mine]), dev) if mine else None
        s.model_list = []
        for g in range(K):
            if g not in mine:
                s.model_list.append(_RemoteModel(shared))
                continue
            m = MF.wrap(merged, Q[mine.index(g)])
            m.user_mat.weight = shared
            if R > 1:
                rows = (len(train_index[g]), d)
                m.checkpoints = [(kn.upload_table(table(f'ckpt{g}_{r}_P', rows), dev),
                                  kn.upload_table(table(f'ckpt{g}_{r}_Q', (s.n_item, d)), dev)) for r in range(R)]
            s.model_list.append(m)
        if s._use_fit():
            tab = st.load_array(state_dir, 'combine')
            if tab.shape != (K, K + 1):
                raise ValueError(f"{state_dir}/combine.npy is {tab.shape}, expected ({K}, {K + 1})")
            s.combination = combination_from(np.ascontiguousarray(tab[:, :K]), np.ascontiguousarray(tab[:, K]),
                                             s._item_tables_in_shard_order(), st.load_array(state_dir, 'combine_gram'))
        return s

    def effective_request(self, users=(), pairs=()):
        """(users int64 [n], pairs int64 [n, 2]) of a deletion request, validated (sisa_state.validate_request), sorted,
        unique and minus what the ledger holds: deleted users, deleted pairs and pairs of deleted users."""
        from . import sisa_state as st
        u, p = st.validate_request(users, pairs, self.n_user, self.n_item)
        return st.effective_request(u, p, self.deleted_users, self.deleted_pairs)

    def retained_data(self, users=(), pairs=()):
        """(train loaders, test loaders, test loader) of the training file minus the ledger's deletions and the given
        ones, read slice-major as the state was trained; ValueError when the reader's count-sorted grouping is not
        the state's train_index (the training file changed)."""
        from . import sisa_state as st
        if self.source is None:
            raise ValueError("Sisa.retained_data needs Sisa.source: the training data the model was learned from")
        du, dp = st.ledger_union(self.deleted_users, self.deleted_pairs,
                                 *st.validate_request(users, pairs, self.n_user, self.n_item))
        tl, sl, total, train_index = st.read_retained(self.source, self.n_user, self.n_group, self.slices, self.batch,
                                                      du, dp, self.device)
        st.check_train_index(train_index, self.group_index)
        return tl, sl, total

    def record_deletions(self, users=(), pairs=()):
        """Add an applied request to the ledger."""
        from . import sisa_state as st
        u, p = st.validate_request(users, pairs, self.n_user, self.n_item)
        self.deleted_users, self.deleted_pairs = st.ledger_union(self.deleted_users, self.deleted_pairs, u, p)
        self.requests += 1

    def apply_request(self, users=(), pairs=(), train_dlist=None, test_dlist=None, test_data=None, verbose=0,
                      save_dir=''):
        """Unlearn a deletion request: deleted users and deleted (user, item) ratings.  Only the effective request
        (effective_request: minus the ledger) is routed, so shards touched only by earlier requests are not retrained;
        the retained data is the training file minus the ledger and the request (retained_data, read here unless the
        loaders are given).  Runs unlearn, then adds the request to the ledger.  Returns the effective request; when
        it is empty nothing is retrained and the model and the ledger stay as they were."""
        from ..config import routed_users
        users, pairs = self.effective_request(users, pairs)
        if len(users) == 0 and len(pairs) == 0:
            self.retrain_gid = set()
            self.first_slice = np.full(self.n_group, self.slices, dtype=np.int32)
            return users, pairs
        if train_dlist is None:
            train_dlist, test_dlist, test_data = self.retained_data(users, pairs)
        self.unlearn(self.model_list, train_dlist, test_dlist, test_data, routed_users(users, pairs), verbose, save_dir)
        self.record_deletions(users, pairs)
        return users, pairs
