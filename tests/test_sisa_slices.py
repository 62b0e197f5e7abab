"""SISA slicing (Sisa.slices = R > 1): each shard trains in R stages over a growing prefix of its slices and keeps the
weights before every stage, so an unlearn retrains a shard only from its first affected slice.

The file restates the definition on top of the unchanged oracle/sisa.py and oracle/mf.py: slice assignment,
slice-major record order, first-affected-slice routing, the stage epochs e' and the stage chain (mf_train from the
previous stage's weights, fresh momentum and StepLR, the keyed Feistel order over the prefix).  CPU: the restatement
against a plain row loop, the host ingest against it, the CLI flag.  GPU: the device ingest against the host split,
a sliced learn against the stage chain, unlearn against a sliced learn on the retained data (bit for bit where the
rounds hold the same shards, within the training tolerances otherwise), the fitted combination and recommend after a
sliced unlearn, several ranks as threads, and the CLI end to end."""
import math
import os
import threading

import numpy as np
import pandas as pd
import pytest

from oracle import mf as omf
from oracle import sisa as osisa

K_TOY = 3


# ------------------------------------------------------------------------------ restatement of the definition
def slice_of_users(group_index, n_user, R):
    """{user: (group, slice)}: a user belongs to the first group listing it; its slice is row * R // m_g."""
    out = {}
    for g, ids in enumerate(group_index):
        m = len(ids)
        for row, u in enumerate(ids):
            if int(u) not in out:
                out[int(u)] = (g, row * R // m)
    return out


def slice_major(kept, group_index, R):
    """The retained rows of every group (oracle read_rating, file order) in slice-major order, stable, and the
    slice boundaries [R + 1] of each group."""
    where = slice_of_users(group_index, 0, R)
    out, offs = [], []
    for arr in kept:
        s = np.array([where[int(u)][1] for u in arr[0]], dtype=np.int64)
        order = np.argsort(s, kind='stable')
        out.append(arr[:, order])
        offs.append(np.concatenate([[0], np.cumsum(np.bincount(s, minlength=R))]))
    return out, offs


def first_slices(group_index, routed, R):
    """Per group the least slice holding a routed user; R when the group has none."""
    where = slice_of_users(group_index, 0, R)
    first = [R] * len(group_index)
    for u in routed:
        if int(u) in where:
            g, s = where[int(u)]
            first[g] = min(first[g], s)
    return first


def stage_epochs_ref(E, R):
    return max(1, math.ceil(2 * E / (R + 1)))


def stage_chain(P0, Q0, u, i, r, off, R, E, shard_id, seed=42, batch=3000, start=0, ckpt=None):
    """Stages start+1 .. R of one shard (mf_train per stage on the prefix of slices 0..j-1, from the previous stage's
    weights); ckpt: the checkpoint list to continue (start > 0).  Returns (checkpoints [R] of (P, Q), P, Q, losses)."""
    E1 = stage_epochs_ref(E, R)
    ck = list(ckpt) if ckpt is not None else [None] * R
    P, Q = (P0, Q0) if start == 0 else ck[start]
    ck[0] = (P0, Q0) if start == 0 else ck[0]
    losses = []
    for j in range(start + 1, R + 1):
        n = int(off[j])
        perms = [omf.feistel_perm(n, omf.perm_key(seed, shard_id, ep)) for ep in range(E1)]
        if n:
            P, Q, _, _, ls = omf.mf_train(P, Q, u[:n], i[:n], r[:n].astype(np.float32), perms, batch, E1)
        else:
            ls = [0.0] * E1
        losses.append(ls)
        if j < R:
            ck[j] = (P, Q)
    return ck, P, Q, losses


def _toy_frames(toy):
    tr = pd.DataFrame({0: toy["train"][0], 1: toy["train"][1], 2: toy["train"][2]})
    te = pd.DataFrame({0: toy["test"][0], 1: toy["test"][1], 2: toy["test"][2]})
    return tr, te


# ------------------------------------------------------------------------------ CPU
def test_restatement_matches_a_row_loop_and_the_product_maps():
    """Slice assignment, slice-major order, routing and e' of the restatement against a plain loop, and the product's
    composite owner map (read._slice_owner) and host routing (Sisa._first_slices) against the restatement."""
    from ultrare_b200.method.sisa import Sisa, _owner_maps, stage_epochs
    from ultrare_b200.read import _slice_owner
    rng = np.random.default_rng(3)
    n_user = 400
    perm = rng.permutation(n_user)
    groups = [perm[:7].tolist(), perm[7:150].tolist(), perm[150:390].tolist()]        # users 390.. in no group
    for R in (1, 2, 3, 8, 32):
        where = slice_of_users(groups, n_user, R)
        for g, ids in enumerate(groups):
            for row, u in enumerate(ids):
                assert where[u] == (g, math.floor(row * R / len(ids)))
        owner = np.full(n_user, -1, dtype=np.int32)
        for g in range(len(groups) - 1, -1, -1):
            owner[np.asarray(groups[g])] = g
        comp = _slice_owner(owner, groups, R)
        want = np.array([where[u][0] * R + where[u][1] if u in where else -1 for u in range(n_user)])
        assert np.array_equal(comp, want)
        # slice-major: stable by slice within the group
        u = rng.integers(0, 390, 5000)
        arr = np.stack([u, rng.integers(0, 50, 5000), rng.integers(1, 6, 5000)]).astype(np.float64)
        kept = [arr[:, np.isin(u, g)] for g in groups]
        got, offs = slice_major(kept, groups, R)
        for g, (a, o) in enumerate(zip(got, offs)):
            rows = []
            for s in range(R):
                rows += [c for c in range(kept[g].shape[1]) if where[int(kept[g][0, c])][1] == s]
            assert np.array_equal(a, kept[g][:, rows]) and o[-1] == kept[g].shape[1]
        # routing
        s = Sisa.__new__(Sisa)
        s.slices, s.n_user, s.n_group, s.group_index = R, n_user, len(groups), groups
        s._owner_np, s._row_of_np = _owner_maps(groups, n_user, 'cpu')[:2]
        for routed in ([], [perm[3]], perm[[5, 100, 200, 395]].tolist(), rng.integers(-3, n_user + 5, 60).tolist()):
            loop = [R] * len(groups)
            for x in routed:
                for g, ids in enumerate(groups):
                    if x in ids:
                        loop[g] = min(loop[g], ids.index(x) * R // len(ids))
                        break
            assert first_slices(groups, routed, R) == loop
            assert s._first_slices(np.asarray(routed, dtype=np.int64)).tolist() == loop
    for E in range(1, 61):
        for R in range(1, 33):
            want = max(1, -(-2 * E // (R + 1)))
            assert stage_epochs(E, R) == stage_epochs_ref(E, R) == want
        assert stage_epochs(E, 1) == E


@pytest.mark.parametrize("R", [1, 3, 8])
def test_host_ingest_is_slice_major(toy, R, monkeypatch, tmp_path):
    """readRating(n_slice=R) and Instance._read_data under URE_HOST_INGEST=1: every shard's rows equal the oracle's
    retained rows in slice-major order; the test sets and the grouping are unchanged."""
    from ultrare_b200.read import readRating
    tr, te = _toy_frames(toy)
    n_user = toy["n_user"]
    del_user = np.random.RandomState(0).choice(n_user, 30, replace=False).tolist()
    got, idx = readRating(tr, n_user, 5, del_user, [], K_TOY, osisa.uniform_groups(n_user, K_TOY), 'a', R)
    kept, gidx = osisa.read_rating(*toy["train"], n_user, 5, del_user, K_TOY, osisa.uniform_groups(n_user, K_TOY), 'a')
    assert [list(g) for g in idx] == [list(g) for g in gidx]
    want, _ = slice_major(kept, gidx, R)
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    unsliced, _ = readRating(tr, n_user, 5, del_user, [], K_TOY, osisa.uniform_groups(n_user, K_TOY), 'a')
    for a, b in zip(got, unsliced):
        assert a.shape == b.shape
    from test_unlearn_interactions import _toy_env
    cfg, _, _ = _toy_env(tmp_path, monkeypatch)
    monkeypatch.setenv('URE_HOST_INGEST', '1')
    ins = cfg.Instance(cfg.InsParam("toy", 1, 1, [32], K_TOY, 2, "rand"))
    ins.slices = R
    train, train_index, test, _ = ins._read_data(True, K_TOY, [], R)
    ftr = pd.read_csv(ins.param.train_dir, header=None)
    fte = pd.read_csv(ins.param.test_dir, header=None)
    kept, gidx = osisa.read_rating(ftr[0].values, ftr[1].values, ftr[2].values, ins.param.n_user, 5,
                                   ins.param.del_user, K_TOY, osisa.uniform_groups(ins.param.n_user, K_TOY), 'a')
    want, _ = slice_major(kept, gidx, R)
    for ds, b in zip(train, want):
        assert np.array_equal(ds._raw, b)
    tk, _ = osisa.read_rating(fte[0].values, fte[1].values, fte[2].values, ins.param.n_user, 5, [], K_TOY,
                              train_index, 'r')
    for ds, b in zip(test, tk):
        assert np.array_equal(ds._raw, b)


def test_host_ingest_rejects_more_than_254_bins(toy):
    from ultrare_b200.read import readRating
    tr, _ = _toy_frames(toy)
    with pytest.raises(ValueError, match="254"):
        readRating(tr, toy["n_user"], 5, [], [], 85, [], 'r', 3)
    out, _ = readRating(tr, toy["n_user"], 5, [], [], 127, [], 'r', 2)
    assert sum(a.shape[1] for a in out) == len(tr)


def test_cli_slices_flag():
    from ultrare_b200.main import _checked, parser
    assert parser.parse_args([]).slices == 1
    assert _checked(parser.parse_args(['--slices', '4', '--group', '3'])).slices == 4
    assert _checked(parser.parse_args(['--slices', '32', '--epoch-eval', 'none'])).slices == 32
    for bad in (['--slices', '0'], ['--slices', '33'], ['--slices', '4', '--epoch-eval', 'faithful'],
                ['--slices', '2', '--group', '0']):
        with pytest.raises(AssertionError):
            _checked(parser.parse_args(bad))
    _checked(parser.parse_args(['--slices', '1', '--group', '0', '--epoch-eval', 'faithful']))


# ------------------------------------------------------------------------------ GPU helpers
def _dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


class _Param:
    def __init__(self, epochs, n_user=1508, n_item=2071):
        self.n_user, self.n_item, self.k, self.lam = n_user, n_item, 16, 0.1
        self.seed, self.lr, self.lr_decay, self.momentum = 42, 0.001, 0.95, 0.9
        self.epochs, self.batch = epochs, 3000


def _inputs(toy, K, R, del_user=(), del_rating=(), device=False):
    """(train loaders, test loaders, test loader, group_index) of the toy data minus the deletions, read slice-major."""
    from ultrare_b200.read import RatingData, loadData, readRating, readRatingDevice
    tr, te = _toy_frames(toy)
    n_user = toy["n_user"]
    groups = osisa.uniform_groups(n_user, K)
    if device:
        trr, idx, _ = readRatingDevice(tr, n_user, 5, list(del_user), list(del_rating), K, groups, 'a', n_slice=R)
        tl = [loadData(d, 3000, 1, True) for d in trr]
    else:
        trr, idx = readRating(tr, n_user, 5, list(del_user), list(del_rating), K, groups, 'a', R)
        tl = [loadData(RatingData(a), 3000, 1, True) for a in trr]
    ter, _ = readRating(te, n_user, 5, [], [], K, idx)
    sl = [loadData(RatingData(a), 3000, 1, False) for a in ter]
    total = loadData(RatingData(np.hstack(ter)), 3000, 1, False)
    return tl, sl, total, idx


def _sisa(K, idx, R, E=2, combine='mean'):
    from ultrare_b200.method.sisa import Sisa
    s = Sisa(_Param(E), 'mf', K, idx)
    s.epoch_eval = 'final'
    s.slices = R
    s.combine = combine
    return s


def _snapshot(s):
    """Host copies of what a pass leaves: merged user table, item tables, every local shard's checkpoints."""
    models = s.model_list
    return dict(P=models[0].user_mat.weight.data.cpu().numpy().copy(),
                Q=[m.item_mat.weight.data.cpu().numpy().copy() for m in models],
                ck=[[(a.cpu().numpy().copy(), b.cpu().numpy().copy()) for a, b in m.checkpoints] for m in models],
                log=dict(s.final_log))


def _learn(toy, K, R, del_user=(), del_rating=(), E=2, combine='mean'):
    tl, sl, total, idx = _inputs(toy, K, R, del_user, del_rating)
    s = _sisa(K, idx, R, E, combine)
    s.learn(tl, sl, total, 0, '')
    return s, idx


def _unlearn(toy, s_before, idx, R, del_user=(), del_rating=(), routed=None, E=2, combine='mean', prev=()):
    from ultrare_b200.config import routed_users
    tl, sl, total, _ = _inputs(toy, len(idx), R, list(prev) + list(del_user), del_rating)
    s = _sisa(len(idx), idx, R, E, combine)
    users = routed_users(list(del_user), np.asarray(del_rating).reshape(-1, 2)) if routed is None else routed
    s.unlearn(list(s_before.model_list), tl, sl, total, users, 0, '')
    return s, tl


def _users_at_slice(idx, R, a, shards):
    """One user per listed shard whose slice is a."""
    return [int(idx[g][-(-a * len(idx[g]) // R)]) for g in shards]


# ------------------------------------------------------------------------------ GPU: ingest
@pytest.mark.gpu
def test_device_ingest_matches_host_split(toy):
    """readRatingDevice(n_slice=R) against readRating(n_slice=R): records bit-equal to the host rows, slice offsets,
    host views; a group smaller than R (empty slices), a slice whose users are all deleted, rating deletions,
    K * R = 254, and a clear error at 255."""
    dev = _dev()
    from ultrare_b200 import kernels as kn  # noqa: F401
    from ultrare_b200.read import readRating, readRatingDevice
    tr, _ = _toy_frames(toy)
    n_user = toy["n_user"]
    perm = np.random.RandomState(5).permutation(n_user)
    groups = [perm[:5].tolist(), perm[5:700].tolist(), perm[700:].tolist()]
    R = 8
    g1 = groups[1]
    gone = [u for row, u in enumerate(g1) if row * R // len(g1) == 2]          # every user of slice 2 of group 1
    rows = np.random.RandomState(1).choice(len(tr), 400, replace=False)
    pairs = np.stack([tr[0].values[rows], tr[1].values[rows]], 1).astype(np.int64)
    cases = [(groups, R, [], []), (groups, R, gone + perm[900:950].tolist(), pairs), (groups, 3, [], pairs),
             ([perm[i::127].tolist() for i in range(127)], 2, perm[:40].tolist(), [])]
    for grp, R_, du, dr in cases:
        host, hidx = readRating(tr, n_user, 5, du, dr, len(grp), grp, 'r', R_)
        ds, didx, total = readRatingDevice(tr, n_user, 5, du, dr, len(grp), grp, 'r', device=dev, n_slice=R_)
        assert [list(g) for g in didx] == [list(g) for g in hidx]
        where = slice_of_users(hidx, n_user, R_)
        for g, (d, h) in enumerate(zip(ds, host)):
            rec = d.records(dev).cpu().numpy()
            assert np.array_equal(rec[:, 0], h[0].astype(np.int32)) and np.array_equal(rec[:, 1], h[1].astype(np.int32))
            assert np.array_equal(rec[:, 2].view(np.float32), h[2].astype(np.float32))
            s = np.array([where[int(u)][1] for u in h[0]], dtype=np.int64)
            assert np.array_equal(d.slice_off, np.concatenate([[0], np.cumsum(np.bincount(s, minlength=R_))]))
            assert np.array_equal(d.users, h[0].astype(int)) and np.array_equal(d._raw, h)
        assert len(total) == sum(h.shape[1] for h in host)
    # the tiny group has empty slices, the deleted slice is empty
    ds, _, _ = readRatingDevice(tr, n_user, 5, gone, [], 3, groups, 'r', device=dev, n_slice=R)
    assert (np.diff(ds[0].slice_off) == 0).sum() >= R - 5 and ds[1].slice_off[3] == ds[1].slice_off[2]
    with pytest.raises(ValueError, match="254"):
        readRatingDevice(tr, n_user, 5, [], [], 85, [], 'r', device=dev, n_slice=3)


# ------------------------------------------------------------------------------ GPU: learn vs the stage chain
@pytest.mark.gpu
def test_sliced_learn_matches_the_stage_chain(toy):
    """A sliced learn (K = 3, R = 3, E = 2: one epoch per stage) against the stage chain of mf_train from the
    model's own initial checkpoint: every checkpoint and the final tables within 1e-4, the losses within 1e-3."""
    _dev()
    K, R, E = K_TOY, 3, 2
    s, idx = _learn(toy, K, R, E=E)
    kept, _ = osisa.read_rating(*toy["train"], toy["n_user"], 5, [], K, osisa.uniform_groups(toy["n_user"], K), 'a')
    arrs, offs = slice_major(kept, idx, R)
    row_of = s._row_of_np
    assert s.timing['rounds'] == R and s.timing['stage_epochs'] == stage_epochs_ref(E, R)
    assert s.timing['trained_interactions'] == sum(int(o[j]) for o in offs for j in range(1, R + 1)) * \
        stage_epochs_ref(E, R)
    losses = np.asarray(s.log['train_loss'])
    assert len(losses) == K * R * stage_epochs_ref(E, R)
    per = R * stage_epochs_ref(E, R)
    for g in range(K):
        m = s.model_list[g]
        P0, Q0 = (t.cpu().numpy() for t in m.checkpoints[0])
        a = arrs[g]
        ck, P, Q, ls = stage_chain(P0, Q0, row_of[a[0].astype(np.int64)], a[1].astype(np.int64), a[2], offs[g], R, E,
                                   g + 1)
        for r in range(1, R):
            assert np.abs(m.checkpoints[r][0].cpu().numpy() - ck[r][0]).max() < 1e-4
            assert np.abs(m.checkpoints[r][1].cpu().numpy() - ck[r][1]).max() < 1e-4
        own = np.asarray(idx[g])
        assert np.abs(m.user_mat.weight.data.cpu().numpy()[own] - P).max() < 1e-4
        assert np.abs(m.item_mat.weight.data.cpu().numpy() - Q).max() < 1e-4
        np.testing.assert_allclose(losses[g * per:(g + 1) * per], np.concatenate(ls), rtol=1e-3)
    assert np.isfinite(s.final_log['total_rmse'])


# ------------------------------------------------------------------------------ GPU: exactness
def _assert_same(a, b, exact):
    cmp = (lambda x, y: np.array_equal(x, y)) if exact else (lambda x, y: np.abs(x - y).max() < 1e-4)
    assert cmp(a['P'], b['P'])
    for x, y in zip(a['Q'], b['Q']):
        assert cmp(x, y)
    for cx, cy in zip(a['ck'], b['ck']):
        for (p1, q1), (p2, q2) in zip(cx, cy):
            assert cmp(p1, p2) and cmp(q1, q2)
    for key in ('total_rmse', 'total_ndcg', 'total_hr'):
        assert a['log'][key] == pytest.approx(b['log'][key], rel=1e-12 if exact else 1e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["first", "middle", "last"])
def test_unlearn_at_one_slice_in_every_shard_is_bit_identical_to_learning_without(toy, where):
    """One deleted user per shard, all at the same slice a: the unlearn's rounds hold every shard with the record
    counts of a sliced learn on the retained data, so tables, checkpoints and merged table are bit-identical (the
    metrics to 1e-12: fp64 atomics); trained interactions = the formula's count; Sisa(slices=1) = the default."""
    _dev()
    K, R, E = K_TOY, 4, 3
    a = {"first": 0, "middle": R // 2, "last": R - 1}[where]
    full, idx = _learn(toy, K, R, E=E)
    du = _users_at_slice(idx, R, a, range(K))
    assert first_slices(idx, du, R) == [a] * K
    un, tl = _unlearn(toy, full, idx, R, du, E=E)
    assert un.first_slice.tolist() == [a] * K and un.retrain_gid == set(range(K))
    E1 = stage_epochs_ref(E, R)
    offs = [t.dataset.slice_off if hasattr(t.dataset, 'slice_off') else un._slice_offsets(t.dataset, g)
            for g, t in enumerate(tl)]
    assert un.timing['trained_interactions'] == sum(int(o[j]) for o in offs for j in range(a + 1, R + 1)) * E1
    assert un.timing['rounds'] == R - a
    assert len(un.log['train_loss']) == K * (R - a) * E1
    ref, _ = _learn(toy, K, R, del_user=du, E=E)
    _assert_same(_snapshot(un), _snapshot(ref), exact=True)
    if where == "middle":           # the unsliced default and slices = 1 run the same code
        from ultrare_b200.method.sisa import Sisa
        tl1, sl1, total1, idx1 = _inputs(toy, K, 1)
        outs = []
        for set_one in (False, True):
            s = Sisa(_Param(2), 'mf', K, idx1)
            s.epoch_eval = 'none'
            if set_one:
                s.slices = 1
            s.learn(tl1, sl1, total1, 0, '')
            outs.append((s.model_list[0].user_mat.weight.data.clone(), [m.item_mat.weight.data.clone()
                                                                        for m in s.model_list], s.final_log))
            assert not hasattr(s.model_list[0], 'checkpoints')
        import torch
        assert torch.equal(outs[0][0], outs[1][0]) and all(torch.equal(x, y) for x, y in zip(outs[0][1], outs[1][1]))
        for key in ('total_rmse', 'total_ndcg', 'total_hr'):
            assert outs[0][2][key] == pytest.approx(outs[1][2][key], rel=1e-12)


@pytest.mark.gpu
def test_unlearn_mixed_slices_interactions_and_two_requests_within_tolerance(toy):
    """Within the training tolerances of a sliced learn on the retained data: one affected shard; mixed first slices;
    a 2 % interaction-level set; two successive requests against a learn on the data minus both.  Unaffected shards
    keep their models and checkpoints."""
    _dev()
    K, R, E = K_TOY, 4, 3
    full, idx = _learn(toy, K, R, E=E)
    before = _snapshot(full)
    # one affected shard
    du = _users_at_slice(idx, R, 2, [1])
    un, _ = _unlearn(toy, full, idx, R, du, E=E)
    assert un.first_slice.tolist() == [R, 2, R] and un.timing['rounds'] == 2
    _assert_same(_snapshot(un), _snapshot(_learn(toy, K, R, du, E=E)[0]), exact=False)
    for g in (0, 2):
        assert un.model_list[g].checkpoints is full.model_list[g].checkpoints
        assert np.array_equal(un.model_list[g].item_mat.weight.data.cpu().numpy(), before['Q'][g])
    # mixed first slices, then a second request on top of it
    du1 = _users_at_slice(idx, R, 1, [0]) + _users_at_slice(idx, R, 3, [2])
    full, _ = _learn(toy, K, R, E=E)
    un1, _ = _unlearn(toy, full, idx, R, du1, E=E)
    assert un1.first_slice.tolist() == [1, R, 3]
    _assert_same(_snapshot(un1), _snapshot(_learn(toy, K, R, du1, E=E)[0]), exact=False)
    du2 = _users_at_slice(idx, R, 0, [1])
    un2, _ = _unlearn(toy, un1, idx, R, du2, E=E, prev=du1)
    assert un2.first_slice.tolist() == [R, 0, R]
    _assert_same(_snapshot(un2), _snapshot(_learn(toy, K, R, du1 + du2, E=E)[0]), exact=False)
    # interaction-level deletions: 2 % of the training rows
    tr, _ = _toy_frames(toy)
    rows = np.sort(np.random.RandomState(0).choice(len(tr), int(0.02 * len(tr)), replace=False))
    pairs = np.stack([tr[0].values[rows], tr[1].values[rows]], 1).astype(np.int64)
    full, _ = _learn(toy, K, R, E=E)
    un3, _ = _unlearn(toy, full, idx, R, del_rating=pairs, E=E)
    assert un3.first_slice.tolist() == first_slices(idx, sorted(set(pairs[:, 0].tolist())), R)
    _assert_same(_snapshot(un3), _snapshot(_learn(toy, K, R, del_rating=pairs, E=E)[0]), exact=False)


@pytest.mark.gpu
def test_unlearn_errors(toy):
    """An unlearn whose models hold no checkpoints, or checkpoints for another R, and R > 1 with 'faithful'."""
    _dev()
    K = K_TOY
    full, idx = _learn(toy, K, 2)
    du = _users_at_slice(idx, 2, 0, [0])
    with pytest.raises(RuntimeError, match="checkpoints"):
        _unlearn(toy, full, idx, 4, du)
    tl, sl, total, idx1 = _inputs(toy, K, 1)
    s = _sisa(K, idx1, 1)
    s.learn(tl, sl, total, 0, '')
    with pytest.raises(RuntimeError, match="checkpoints"):
        _unlearn(toy, s, idx, 2, du)
    s = _sisa(K, idx, 2)
    s.epoch_eval = 'faithful'
    with pytest.raises(ValueError, match="epoch_eval"):
        s.learn(*_inputs(toy, K, 2)[:3], 0, '')


# ------------------------------------------------------------------------------ GPU: fit, recommend, ranks
@pytest.mark.gpu
def test_fit_and_recommend_after_sliced_unlearn_and_ranks(toy):
    """combine='fit' after a sliced unlearn equals the float64 oracle fitted on the retained rows; recommend equals the
    oracle top-N; 2 and 3 ranks (threads on one GPU) unlearning from the same learn agree with one GPU."""
    import torch
    from oracle import combine as ocomb
    from oracle import recommend as orec
    from test_combine import _ThreadDist
    from ultrare_b200 import kernels as kn
    from ultrare_b200.method.sisa import Sisa, _RemoteModel
    dev = _dev()
    K, R, E = K_TOY, 4, 2
    n_user = toy["n_user"]
    full, idx = _learn(toy, K, R, E=E, combine='fit')
    keep_P = full.model_list[0].user_mat.weight
    du = np.random.RandomState(0).choice(n_user, 30, replace=False).tolist()
    un, tl = _unlearn(toy, full, idx, R, du, E=E, combine='fit')
    P = un.model_list[0].user_mat.weight.data
    Qs = [m.item_mat.weight.data for m in un.model_list]
    P_h, Q_h = P.cpu().numpy(), [q.cpu().numpy() for q in Qs]
    kept, _ = osisa.read_rating(*toy["train"], n_user, 5, du, K, osisa.uniform_groups(n_user, K), 'a')
    w_o, b_o = ocomb.fit(P_h, Q_h, [(a[0].astype(np.int64), a[1].astype(np.int64), a[2]) for a in kept])
    owner = un._owner_np
    te = np.hstack(osisa.read_rating(*toy["test"], n_user, 5, [], K, idx, 'r')[0])
    rec_te = kn.pack_interactions(te[0].astype(np.int64), te[1].astype(np.int64), te[2].astype(np.float32), dev)
    got, _ = kn.group_score(P, un.combination.T, un.combination.b_slot, un._owner, rec_te)
    want = ocomb.scores(P_h, Q_h, w_o, b_o, owner, te[0].astype(np.int64), te[1].astype(np.int64))
    assert np.abs(got.cpu().numpy() - want).max() <= 1e-4
    items, scores = un.recommend(None, 10, exclude=tl)
    train = np.hstack(kept)
    rec = torch.from_numpy(np.stack([train[0], train[1], train[2], train[2]], 1).astype(np.int32)).to(dev)
    oi, ov = ocomb.topn(P_h, Q_h, un.combination.w, un.combination.b, owner, np.arange(n_user), 10,
                        orec.seen_sets(rec.cpu().numpy(), n_user))
    assert (items.cpu().numpy() == oi).mean() > 0.99
    np.testing.assert_allclose(scores.cpu().numpy(), ov, atol=1e-4)
    one = _snapshot(un)

    lock = threading.Lock()
    for world in (2, 3):
        for m in full.model_list:                  # the learn's state again: unlearn rebinds the shared user table
            m.user_mat.weight = keep_P
        shared = dict(barrier=threading.Barrier(world), slots=[None] * world)
        out, errs = [None] * world, []
        tl2, sl2, total2, _ = _inputs(toy, K, R, du)

        def run(r):
            try:
                sr = _sisa(K, idx, R, E, 'fit')
                sr.dist = _ThreadDist(r, world, shared)
                train_one = sr._train_sliced

                def serial(*a, **k):                # the ranks' training launches one after another
                    with lock:
                        return train_one(*a, **k)
                sr._train_sliced = serial
                models = [m if k % world == r else _RemoteModel(keep_P) for k, m in enumerate(full.model_list)]
                sr.unlearn(models, tl2, sl2, total2, du, 0, '')
                out[r] = (sr.model_list[0].user_mat.weight.data.cpu().numpy(),
                          {k: m.item_mat.weight.data.cpu().numpy() for k, m in enumerate(sr.model_list)
                           if k % world == r}, dict(sr.final_log))
            except BaseException as e:      # noqa: BLE001 -- re-raised below; the other ranks are released
                errs.append(e)
                shared["barrier"].abort()

        th = [threading.Thread(target=run, args=(r,)) for r in range(world)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errs:
            raise errs[0]
        for r, (Pm, Qm, log) in enumerate(out):
            assert np.abs(Pm - one['P']).max() < 1e-4, (world, r)
            for k, q in Qm.items():
                assert np.abs(q - one['Q'][k]).max() < 1e-4, (world, r, k)
            assert log['total_rmse'] == pytest.approx(one['log']['total_rmse'], rel=1e-3)


# ------------------------------------------------------------------------------ GPU: CLI
@pytest.mark.gpu
@pytest.mark.parametrize("deltype", ["rand", "inter"])
def test_cli_slices_end_to_end(cuda_dev, tmp_path, monkeypatch, deltype):
    """--slices 4 --group 3 --grouping rating-ot: the usual artefacts of both passes plus slices.npy (int32 [K], the
    first retrained slice of every shard, 4 = not retrained) equal to the routing restated."""
    from test_unlearn_interactions import _toy_env
    from ultrare_b200.config import routed_users
    from ultrare_b200.main import main
    monkeypatch.setenv('ULTRARE_EPOCH_EVAL', 'faithful')      # restored afterwards; --slices without --epoch-eval: final
    _, _, save = _toy_env(tmp_path, monkeypatch)
    ins = main(['--dataset', 'toy', '--synth', '--deltype', deltype, '--epoch', '2', '--worker', '1', '--verbose', '0',
                '--group', '3', '--grouping', 'rating-ot', '--slices', '4', '--recommend', '5'])
    s = ins.last_sisa
    assert s.slices == 4 and s.epoch_eval == 'final'
    gdir = f'{save}/2/{deltype}/toy_g3'
    for sub in ('MF_rating-ot_sisa_learn', 'MF_rating-ot_sisa_unlearn'):
        assert os.path.exists(f'{gdir}/{sub}/log0.npy') and os.path.exists(f'{gdir}/{sub}/rec5.npy'), sub
    for i in range(1, 4):
        assert os.path.exists(f'{gdir}/MF_rating-ot_sisa_learn/model{i}.pth')
    sl = np.load(f'{gdir}/MF_rating-ot_sisa_unlearn/slices.npy')
    assert sl.dtype == np.int32 and sl.shape == (3,)
    users = routed_users(ins.param.del_user, ins.param.del_rating)
    assert sl.tolist() == first_slices(s.group_index, users, 4)
    assert (sl < 4).any()
    for g in range(3):
        if sl[g] < 4:
            assert os.path.exists(f'{gdir}/MF_rating-ot_sisa_unlearn/model{g + 1}.pth')
    assert not os.path.exists(f'{gdir}/MF_rating-ot_sisa_learn/slices.npy')
