"""B200 mirror of the reference's single-model trainer (method/scratch.py:11-148).

Same constructor and ``train`` signature, same log keys, same on-disk artefacts
(``model{id}.pth``, ``user_mat{id}.npy``, ``item_mat{id}.npy``, ``log{id}.npy``).  The epoch
body is one persistent kernel launch (``baseTrain``) plus the fused evaluation kernels
(``baseTest``); optimiser state stays on the device.
"""
from __future__ import annotations

import time

import numpy as np
import torch
from torch import nn

from .utils import MF, FusedSGD, baseTest, baseTrain, seed_all, _cuda_device


def model_generator(seed: int, id: int, device='cpu') -> torch.Generator:
    """Init-weight generator for model `id` (the reference's init is unseeded; SURVEY.md H8).
    device='cpu' gives device-independent values; a CUDA device draws on the GPU."""
    g = torch.Generator(device=device)
    g.manual_seed(int(seed) * 1000003 + int(id))
    return g


class Scratch(object):
    def __init__(self, param, model_type):
        # model param (reference scratch.py:13-17)
        self.n_user = param.n_user
        self.n_item = param.n_item
        self.k = param.k
        self.lam = param.lam
        self.model_type = model_type
        # training param (scratch.py:20-31; dis_type/attr default as Appendix A2)
        self.seed = param.seed
        self.lr = param.lr
        self.lr_decay = param.lr_decay
        self.momentum = param.momentum
        self.epochs = param.epochs
        self.batch = getattr(param, 'batch', 30000)
        self.loss = getattr(param, 'loss', 'mse')
        if self.loss not in ('mse', 'bpr'):
            raise ValueError(f"loss must be 'mse' or 'bpr', not {self.loss!r}")
        self.device = _cuda_device()
        self.dis_type = getattr(param, 'dis_type', 'nor')
        self.attr = [] if self.dis_type == 'nor' else getattr(param, 'attr', [])
        assert self.dis_type == 'nor', "u2u/d2d regularisers are out of scope (SURVEY.md §2.1 row 14)"
        # log (scratch.py:35-42)
        self.log = {'train_loss': [], 'test_rmse': [], 'test_ndcg': [], 'test_hr': [],
                    'total_rmse': [], 'total_ndcg': [], 'total_hr': [], 'time': []}
        if self.model_type == 'mf':
            self.loss_fn = nn.MSELoss(reduction='sum')
            self.is_rmse = True
        else:
            raise ValueError("only model_type='mf' exists in the reference source (SURVEY.md §2.1 row 17)")

    @staticmethod
    def _no_total(test_total):
        return isinstance(test_total, (list, tuple)) and len(test_total) == 0

    init_on_device = True     # False: host generator (same weights on any device, slower)
    loss = 'mse'              # training objective (param.loss): 'mse' = the reference's, 'bpr' = pairwise ranking

    def _new_model(self, id, user_rows=None):
        gen = model_generator(self.seed, id, self.device if self.init_on_device else 'cpu')
        return MF(self.n_user, self.n_item, self.k, device=self.device, generator=gen, user_rows=user_rows)

    def train(self, train_data, test_data, test_total=[], verbose=1, save_dir='', id=0, given_model=''):
        print('Using device:', self.device)
        seed_all(self.seed)
        if isinstance(given_model, str) and given_model == '':
            model = self._new_model(id)
        else:
            model = given_model.to(self.device)
        opt = FusedSGD(model, lr=self.lr, weight_decay=self.lam, momentum=self.momentum, lr_decay=self.lr_decay,
                       lr_step=50, epochs=self.epochs, perm_seed=self.seed, shard_id=id, loss=self.loss)

        for t in range(self.epochs):
            if verbose == 2:
                print(f'Epoch: [{t+1:>3d}/{self.epochs:>3d}] --------------------')
            epoch_start = time.time()
            train_loss, train_rmse = baseTrain(train_data, model, self.loss_fn, self.is_rmse, opt, self.device,
                                               verbose, self.dis_type, self.attr)
            models = (self.model_list + [model]) if self.__class__.__name__ == 'Sisa' else [model]
            test_rmse, test_ndcg, test_hr = baseTest(test_data, models, self.loss_fn, self.device, verbose)
            if self._no_total(test_total):
                total_rmse, total_ndcg, total_hr = test_rmse, test_ndcg, test_hr
            else:
                total_rmse, total_ndcg, total_hr = baseTest(test_total, models, self.loss_fn, self.device, verbose)
            epoch_time = time.strftime('%H:%M:%S', time.gmtime(time.time() - epoch_start))
            if verbose == 2:
                print('Time:', epoch_time)
            elif verbose == 1:
                msg = (f'Epoch: [{t+1:>2d}/{self.epochs:>2d}] train loss: {train_loss:>.9f},'
                       f' train RMSE: {train_rmse:>.4f}, test RMSE: {test_rmse:>.4f},')
                if not self._no_total(test_total):
                    msg += f' total RMSE: {total_rmse:>.4f},'
                print(msg + ' time:', epoch_time)
            self.log['train_loss'].append(train_loss)
            self.log['test_rmse'].append(test_rmse)
            self.log['test_ndcg'].append(test_ndcg)
            self.log['test_hr'].append(test_hr)
            self.log['time'].append(epoch_time)
            if not self._no_total(test_total):
                self.log['total_rmse'].append(total_rmse)
                self.log['total_ndcg'].append(total_ndcg)
                self.log['total_hr'].append(total_hr)

        self._save(model, save_dir, id)
        return model

    def _save(self, model, save_dir, id):
        """reference scratch.py:131-144."""
        if len(save_dir) > 0:
            torch.save(model.state_dict(), save_dir + '/model' + str(id) + '.pth')
            np.save(save_dir + '/user_mat' + str(id), model.user_mat.weight.detach().cpu().numpy())
            np.save(save_dir + '/item_mat' + str(id), model.item_mat.weight.detach().cpu().numpy())
            np.save(save_dir + '/log' + str(id), self.log)
