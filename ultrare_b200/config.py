"""B200 mirror of the reference's experiment driver (config.py): InsParam and Instance.

Same class names, constructor arguments, attributes, result-directory naming and the two
entry points ``Instance.runFull(is_save, verbose)`` / ``Instance.runGroup(is_save,
learn_type, group_type, n_group, verbose)`` (config.py:182-200).  Defects of the reference
are resolved as SURVEY.md Appendix A lists (A1 del_per is a percentage, A2 dis_type, A11 the
embedding path follows the current del_per/del_type with the literal path as fallback).
The reference always leaves del_rating empty (Appendix A13); here del_type='inter' fills it with deleted
(user, item) ratings, which the training reads drop and whose users' shards are retrained.
"""
from __future__ import annotations

import os
import time
import warnings
from os.path import exists

import numpy as np

from .group import DATA_DIR, SAVE_DIR, Group
from .method.scratch import Scratch
from .method.sisa import Sisa
from .method.utils import recommend, saveObject, topn_metrics
from .read import RatingData, loadData, readRating, readRatingDevice, readSparseMat

DATASETS = {
    # name: (train file, test file, n_user, n_item, batch)   reference config.py:26,40-44
    'ml1m': ('/ml1m/squ0_train.csv', '/ml1m/squ0_test.csv', 6040, 3416, 30000),
    'toy': ('/toy/0_train.csv', '/toy/0_test.csv', 1508, 2071, 3000),
}


def draw_rating_deletions(train_dir, del_per):
    """del_type='inter': int64 [n_del, 2] (user, item) of del_per % of the training file's rows, drawn without
    replacement under np.random.seed(0), in file order."""
    import pandas as pd
    ratings = pd.read_csv(train_dir, header=None, sep=',')
    n = len(ratings)
    np.random.seed(0)
    rows = np.sort(np.random.choice(n, int(del_per / 100 * n), replace=False))
    return np.stack([ratings[0].values[rows], ratings[1].values[rows]], axis=1).astype(np.int64)


def routed_users(del_user, del_rating):
    """The users whose shards an unlearn pass retrains (config.py:190-193): del_user, then the users of del_rating
    that it does not hold, in order of first appearance.  Exactly list(del_user) when del_rating is empty."""
    out = list(del_user)
    if len(del_rating) == 0:
        return out
    users = np.asarray(del_rating)[:, 0]
    _, first = np.unique(users, return_index=True)
    new = users[np.sort(first)]
    return out + new[~np.isin(new, np.asarray(out))].tolist()


def save_recommendations(save_dir, N, items, scores, test_data):
    """rec{N}.npy (int32 [n_user, N] item ids), rec{N}_score.npy (fp32) and rec{N}_metrics.npy (fp64 [4]: HR@N,
    Recall@N, NDCG@N over the whole catalogue, users counted) into the pass's save directory."""
    from . import dist as udist
    met = topn_metrics(items, None, test_data, N)
    print(f'Top-{N} over the catalogue - HR: {met["hr"]:>.4f}, Recall: {met["recall"]:>.4f}, '
          f'NDCG: {met["ndcg"]:>.4f} ({met["users"]} users)')
    if len(save_dir) > 0 and udist.get().rank == 0:
        np.save(f'{save_dir}/rec{N}', items.cpu().numpy())
        np.save(f'{save_dir}/rec{N}_score', scores.cpu().numpy())
        np.save(f'{save_dir}/rec{N}_metrics',
                np.array([met['hr'], met['recall'], met['ndcg'], met['users']], dtype=np.float64))


def check_out_dir(out_dir):
    """A request run writes into a directory that does not exist yet or is empty: it never mixes with, or
    overwrites, another run's files."""
    if os.path.exists(out_dir) and (not os.path.isdir(out_dir) or os.listdir(out_dir)):
        raise ValueError(f"the output directory {out_dir} exists and is not empty; a request run writes into a new or "
                         "empty directory")


def run_request(state_dir, out_dir, users=(), pairs=(), recommend_n=0, verbose=1):
    """Apply one deletion request to the SISA state in `state_dir` (Sisa.load_state, Sisa.apply_request) and write
    into `out_dir`: the artefacts of an unlearn pass (log*.npy; user_mat*, item_mat*, model*.pth of the retrained
    shards; combine.npy; slices.npy; rec{N}*.npy), deletion.npy (the effective request, sisa_state.deletion_table)
    and state/, the updated state.  The input state is only read.  Returns the Sisa."""
    from . import dist as udist
    from .method import sisa_state as st
    d = udist.get()
    check_out_dir(out_dir)
    d.barrier()
    print(state_dir, 'deletion request begin:')
    model = Sisa.load_state(state_dir)
    users, pairs = model.effective_request(users, pairs)
    os.makedirs(out_dir, exist_ok=True)
    if len(users) == 0 and len(pairs) == 0:
        print('The request holds only deletions the state has already applied: no shard is retrained, '
              'the state is unchanged')
    else:
        print(f'Effective request: {len(users)} users, {len(pairs)} ratings')
        train_dlist, test_dlist, test_data = model.retained_data(users, pairs)
        model.apply_request(users, pairs, train_dlist, test_dlist, test_data, verbose, out_dir)
        if model.slices > 1 and d.rank == 0:
            np.save(out_dir + '/slices', model.first_slice.astype(np.int32))
        if recommend_n > 0:
            save_recommendations(out_dir, recommend_n, *model.recommend(None, recommend_n, exclude=train_dlist),
                                 test_data)
    if d.rank == 0:
        np.save(out_dir + '/deletion', st.deletion_table(users, pairs))
    model.save_state(out_dir + '/state')
    print('End of request', out_dir)
    return model


class InsParam(object):
    # training objective of every model (Scratch.loss / Sisa.loss, main.py --loss): 'mse' = the reference's squared
    # rating error, 'bpr' = pairwise ranking with sampled negatives (implicit feedback)
    loss = 'mse'

    def __init__(self, dataset='toy', epochs=50, n_worker=24, layers=[32], n_group=2, del_per=2, del_type='test'):
        # model param (config.py:19-21)
        self.k = 16
        self.lam = 0.1
        self.layers = layers
        # training param (config.py:24-31)
        self.seed = 42
        self.n_worker = n_worker
        self.batch = 3000 if dataset == 'toy' else 30000
        self.lr = 0.001
        self.lr_decay = 0.95
        self.momentum = 0.9
        self.epochs = epochs
        self.n_group = n_group
        self.dis_type = 'nor'            # Appendix A2
        self.attr = []
        # dataset-varied param (config.py:34-49)
        self.del_rating = []
        self.dataset = dataset
        self.max_rating = 5
        self.del_per = del_per
        self.del_type = del_type
        self.del_user = np.array([], dtype=np.int64)
        if dataset in DATASETS:
            tr, te, self.n_user, self.n_item, self.batch = DATASETS[dataset]
            self.train_dir = DATA_DIR + tr
            self.test_dir = DATA_DIR + te
            if self.del_type == 'rand':
                np.random.seed(0)
                n_del = int(self.del_per / 100 * self.n_user)      # Appendix A1
                self.del_user = np.random.choice(self.n_user, n_del, replace=False)
            elif self.del_type == 'inter':
                self.del_rating = draw_rating_deletions(self.train_dir, self.del_per)

    def info(self):
        print(self.dataset, '-----------')
        print('Path of training data:', self.train_dir)
        print('Path of testing data:', self.test_dir)
        print('Number of users:', self.n_user)
        print('Number of items:', self.n_item)


class Instance(object):
    recommend_n = 0          # > 0: every pass also writes top-N recommendations and their metrics (main.py --recommend)
    combine = 'mean'         # how the SISA passes combine the shard models: 'mean' or 'fit' (Sisa.combine, --combine)
    slices = 1               # SISA slices per shard (Sisa.slices, --slices); the training reads come slice-major
    save_state = False       # every SISA pass also writes its model as state/ in its directory (--save-state)

    def __init__(self, param):
        self.param = param
        prefix = '/test/' if self.param.del_type == 'test' else '/' + str(self.param.del_per) + '/' + self.param.del_type + '/'
        self.name = prefix + self.param.dataset + '_g' + str(self.param.n_group)
        if self.param.loss == 'bpr':           # BPR runs keep their artefacts apart from the MSE runs'
            self.name += '_bpr'
        param_dir = SAVE_DIR + self.name
        os.makedirs(param_dir, exist_ok=True)
        saveObject(param_dir + '/param', self.param)
        arr = np.empty(2, dtype=object)
        arr[0], arr[1] = self.param.del_user, self.param.del_rating
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            np.save(param_dir + '/deletion', arr)
        self.timing = {}

    # read raw data (config.py:80-96)
    def _read(self, is_del=False, n_group=1, group_index=[], n_slice=1):
        del_user = self.param.del_user if is_del == True else []
        del_rating = self.param.del_rating if is_del == True else []
        train_rating, train_index = readRating(self.param.train_dir, self.param.n_user, self.param.max_rating,
                                               del_user, del_rating, n_group, group_index, 'a', n_slice)
        test_rating, _ = readRating(self.param.test_dir, self.param.n_user, self.param.max_rating,
                                    [], [], n_group, train_index)
        return train_rating, train_index, test_rating

    # the same read with the filter/split on the GPU: RatingData objects instead of arrays (read.readRatingDevice);
    # URE_HOST_INGEST=1 keeps the host split of `_read`
    def _read_data(self, is_del=False, n_group=1, group_index=[], n_slice=1):
        import torch
        if os.environ.get('URE_HOST_INGEST', '0') == '1' or not torch.cuda.is_available():
            train_rating, train_index, test_rating = self._read(is_del, n_group, group_index, n_slice)
            return ([RatingData(r) for r in train_rating], train_index, [RatingData(r) for r in test_rating],
                    RatingData(np.hstack(test_rating)))
        del_user = self.param.del_user if is_del == True else []
        del_rating = self.param.del_rating if is_del == True else []
        train, train_index, _ = readRatingDevice(self.param.train_dir, self.param.n_user, self.param.max_rating,
                                                 del_user, del_rating, n_group, group_index, 'a', n_slice=n_slice)
        test, _, test_total = readRatingDevice(self.param.test_dir, self.param.n_user, self.param.max_rating,
                                               [], [], n_group, train_index)
        return train, train_index, test, test_total

    def _save_dir(self, is_save, saving_name):
        if is_save != True:
            return ''
        save_dir = SAVE_DIR + self.name + '/' + saving_name
        os.makedirs(save_dir, exist_ok=True)
        return save_dir

    # sub function of self.runFull (config.py:99-120)
    def _full(self, is_save, saving_name, model_type='mf', is_del=False, verbose=1):
        print(self.name, saving_name, 'begin:')
        train, _, test, _ = self._read_data(is_del)
        train_data = loadData(train[0], self.param.batch, self.param.n_worker)
        test_data = loadData(test[0], self.param.batch, self.param.n_worker, False)
        save_dir = self._save_dir(is_save, saving_name)
        model = Scratch(self.param, model_type)
        trained = model.train(train_data, test_data, [], verbose, save_dir)
        if self.recommend_n > 0:
            self._save_recommendations(save_dir, *recommend([trained], None, self.recommend_n, exclude=train_data),
                                       test_data)
        print('End of training', self.name, saving_name)
        print()
        return model

    def _user_mat_path(self):
        cands = [SAVE_DIR + '/' + str(self.param.del_per) + '/' + self.param.del_type + '/' + self.param.dataset
                 + '_g0/MF_full_train/user_mat0.npy',
                 "{}/2/rand/ml1m_g0/MF_full_train/user_mat0.npy".format(SAVE_DIR)]          # config.py:132
        for c in cands:
            if exists(c):
                return c
        raise FileNotFoundError("user_mat0.npy not found (run `--group 0` first, config.py:132): " + cands[0])

    def _group_index(self, group_type, n_group):
        """The user grouping of config.py:126-134: [] for 'uniform' (readRating draws it), else Group.grouping.
        'emb-ot' clusters the user table of a `--group 0` run (user_mat0.npy); 'rating-ot' clusters the users' rows of
        the whole training file (readSparseMat, config.py:130) and needs no earlier run.
        One process per GPU (torchrun): rank 0 alone computes (or loads) the grouping and writes the cache file;
        every rank then holds the SAME group_index -- the centroid sums are order-dependent fp64 atomics, so two
        ranks clustering on their own could end with different labels and different owner maps."""
        if group_type == 'uniform':
            return []
        from . import dist as udist
        d = udist.get()
        t0 = time.time()
        group_index = None
        if d.rank == 0:
            if group_type.startswith('rating'):
                X = readSparseMat(self.param.train_dir, self.param.n_user, self.param.n_item, self.param.max_rating)
                grp = Group(X, self.param.dataset)
            else:
                user_mat = np.load(self._user_mat_path(), allow_pickle=True)
                shape = type('Shape', (), {'shape': (self.param.n_user, self.param.n_item)})()   # shapes only
                grp = Group(shape, self.param.dataset, user_mat)
            group_index = grp.grouping(self.param.dataset, n_group, group_type, verbose=False)
        group_index = d.broadcast_object(group_index, src=0)
        self.timing['grouping_s'] = time.time() - t0
        return group_index

    # sub function of self.runGroup (config.py:123-174)
    def _group(self, model_list, is_save, learn_type, saving_name, model_type='mf',
               is_del=False, group_type='uniform', n_group=5, verbose=1):
        print(self.name, saving_name, 'begin:')
        group_index = self._group_index(group_type, n_group)

        train, train_index, test, test_total = self._read_data(is_del, n_group, group_index, self.slices)

        train_dlist, test_dlist = [], []
        assert learn_type in ['sisa']
        for i in range(n_group):
            train_dlist.append(loadData(train[i], self.param.batch, self.param.n_worker))
            test_dlist.append(loadData(test[i], self.param.batch, self.param.n_worker, False))
        test_data = loadData(test_total, self.param.batch, self.param.n_worker, False)         # config.py:144-148

        save_dir = self._save_dir(is_save, saving_name)
        model = Sisa(self.param, model_type, n_group, train_index)
        model.combine = self.combine
        model.slices = self.slices
        model.source = dict(dataset=self.param.dataset, train_file=self.param.train_dir, test_file=self.param.test_dir,
                            max_rating=self.param.max_rating, grouping=group_type, group_index=group_index)
        t0 = time.time()
        if is_del == False:
            model.learn(train_dlist, test_dlist, test_data, verbose, save_dir)
            self.timing['learn_s'] = time.time() - t0
        else:
            del_user = routed_users(self.param.del_user, self.param.del_rating)
            model.unlearn(model_list, train_dlist, test_dlist, test_data, del_user, verbose, save_dir)
            self.timing['unlearn_s'] = time.time() - t0
            if self.slices > 1 and len(save_dir) > 0 and model.dist.rank == 0:
                # int32 [K]: the first retrained slice of every shard (slices = not retrained)
                np.save(save_dir + '/slices', model.first_slice.astype(np.int32))
            if self.save_state:
                model.record_deletions(self.param.del_user, self.param.del_rating)      # the ledger of the state
        if self.recommend_n > 0:
            # seen items: this pass's training data (after the unlearn pass, deleted users' old items are gone)
            self._save_recommendations(save_dir, *model.recommend(None, self.recommend_n, exclude=train_dlist), test_data)
        if self.save_state and len(save_dir) > 0:
            model.save_state(save_dir + '/state')
        self.last_sisa = model
        return model.model_list

    def _save_recommendations(self, save_dir, items, scores, test_data):
        save_recommendations(save_dir, self.recommend_n, items, scores, test_data)

    # ---------------------------------------------------------------- calling functions
    def runFull(self, is_save=True, verbose=1):
        '''model MF (config.py:182-188)'''
        self._full(is_save, 'MF_full_train', 'mf', False, verbose)
        self._full(is_save, 'MF_retrain', 'mf', True, verbose)

    def runGroup(self, is_save=True, learn_type='seq', group_type='uniform', n_group=5, verbose=1):
        '''model MF (config.py:190-200)'''
        saving_name = 'MF_' + group_type + '_' + learn_type + '_learn'
        model_list = self._group([], is_save, learn_type, saving_name, 'mf', False, group_type, n_group, verbose)
        saving_name = 'MF_' + group_type + '_' + learn_type + '_unlearn'
        self._group(model_list, is_save, learn_type, saving_name, 'mf', True, group_type, n_group, verbose)
