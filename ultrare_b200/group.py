"""B200 mirror of the reference's group.py: OT-based user grouping with an on-disk cache.

``Group(rating, dataset, user_mat).grouping(dataset, n_group, var, verbose)`` as in the
reference (group.py:16-66), with its defects resolved as SURVEY.md Appendix A3-A5 lists:
the 'emb-ot' branch reaches ``ot_cluster``; the return value is ALWAYS the list of K
ascending user-id lists (what ``readRating`` consumes, read.py:59); ``val/`` is created and
the ragged list is saved as an object array.
"""
from __future__ import annotations

import os
import warnings
from os.path import abspath, dirname, exists, join

import numpy as np

from .method.utils import ot_cluster

_ROOT = os.environ.get('ULTRARE_ROOT', abspath(join(dirname(__file__), '..')))
DATA_DIR = abspath(join(_ROOT, 'data'))      # reference group.py:9
SAVE_DIR = abspath(join(_ROOT, 'result'))    # reference group.py:10


class Group(object):
    def __init__(self, rating, dataset, user_mat=None):
        self.rating = rating                   # csr_matrix ('rating-ot') or anything with .shape ('emb-ot')
        self.dataset = dataset
        self.user_mat = user_mat
        self.n_user = self.rating.shape[0]
        self.n_item = self.rating.shape[1]

    def grouping(self, dataset='ml1m', n_group=2, var='emb-ot', verbose=True, use_cache=True):
        assert n_group > 1
        label_dir = DATA_DIR + '/' + dataset + '/val/' + var + str(n_group) + '.npy'
        if use_cache and exists(label_dir):                                   # group.py:30-32
            res = np.load(label_dir, allow_pickle=True)
            return [list(map(int, g)) for g in res]

        trans_var, cluster_var = var.strip().split('-')
        assert cluster_var == 'ot', "only '<x>-ot' grouping is reachable from main.py (main.py:64)"
        if trans_var == 'emb':
            points = np.asarray(self.user_mat, dtype=np.float32)
        elif trans_var == 'rating':
            points = self.rating                 # the sparse rating rows, clustered without densifying
        else:
            raise ValueError(var)
        _, label = ot_cluster(points, n_group)                                   # Appendix A3

        if verbose == True:
            print(''.join(f'{i}: {int((label == i).sum())}, ' for i in range(n_group)))

        res = [np.flatnonzero(label == idx).tolist() for idx in range(n_group)]  # group.py:56-58
        os.makedirs(dirname(label_dir), exist_ok=True)                           # Appendix A5
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            arr = np.empty(n_group, dtype=object)
            for idx in range(n_group):
                arr[idx] = res[idx]
            tmp = label_dir + '.tmp%d.npy' % os.getpid()     # atomic: a concurrent reader never sees half a file
            np.save(tmp, arr)
            os.replace(tmp, label_dir)
        return res                                                               # Appendix A4
