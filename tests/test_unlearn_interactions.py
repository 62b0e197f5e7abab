"""Interaction-level unlearning: deleted (user, item) ratings are dropped by the training reads (host filter and the
device partition), their users' shards are retrained, and --deltype inter draws them from the training file."""
import os

import numpy as np
import pandas as pd
import pytest

from oracle import sisa as osisa


def _deletion_pairs(users, items, del_per, seed=0):
    """Restatement of the --deltype inter draw: int64 [n_del, 2] (user, item) of int(del_per/100 * n) training rows
    drawn without replacement (legacy RandomState), in file order."""
    users, items = np.asarray(users), np.asarray(items)
    n = len(users)
    rows = np.sort(np.random.RandomState(seed).choice(n, int(del_per / 100 * n), replace=False))
    return np.stack([users[rows], items[rows]], axis=1).astype(np.int64)


def _read_rating(users, items, ratings, n_user, max_rating=5, del_user=(), n_group=1, group_index=(), sort='r',
                 del_rating=()):
    """oracle.sisa.read_rating with deleted ratings: the group order counts the unfiltered rows, then every row whose
    (int(user), int(item)) is a listed pair is dropped (every copy) before the per-group filter."""
    users, items, ratings = np.asarray(users), np.asarray(items), np.asarray(ratings)
    _, group_index = osisa.read_rating(users, items, ratings, n_user, max_rating, (), n_group, group_index, sort)
    pairs = set((int(p[0]), int(p[1])) for p in del_rating)
    if any(u < 0 or i < 0 for u, i in pairs):
        raise ValueError("del_rating: negative id")
    keep = np.array([(int(u), int(i)) not in pairs for u, i in zip(users, items)], dtype=bool)
    return osisa.read_rating(users[keep], items[keep], ratings[keep], n_user, max_rating, del_user, n_group,
                             group_index, 'r')


def _table(seed=5, n_user=700, n_item=300, n=20000):
    """A ratings table, deleted users, and deleted pairs covering every case the filter must handle."""
    rng = np.random.default_rng(seed)
    u = rng.integers(0, n_user, n)
    i = rng.integers(0, n_item, n)
    r = rng.integers(1, 6, n).astype(np.float64)
    u[100], i[100] = u[50], i[50]                             # a pair that occurs twice in the file
    del_user = [int(x) for x in rng.choice(n_user, 40, replace=False)]
    rows = rng.choice(n, n // 30, replace=False)
    pairs = [np.stack([u[rows], i[rows], r[rows]], 1)]        # a third column, which is ignored
    pairs.append(pairs[0][:25])                               # duplicate pairs
    pairs.append(np.array([[u[50], i[50], 0.0]]))
    pairs.append(np.stack([rng.integers(0, n_user, 30), n_item + rng.integers(0, 50, 30), np.zeros(30)], 1))  # no match
    of_del = np.flatnonzero(np.isin(u, del_user))[:15]
    pairs.append(np.stack([u[of_del], i[of_del], r[of_del]], 1))                  # pairs of deleted users
    pairs.append(np.array([[n_user + 1000, 3, 0.0], [n_user + 7, 0, 0.0]]))       # users outside the owner map
    pairs = np.concatenate(pairs).astype(np.int64)
    return pd.DataFrame({0: u, 1: i, 2: r}), n_user, del_user, pairs


def _brute(df, n_user, del_user, pairs, groups, max_rating=5):
    """Row by row: a row stays in the first group listing its user unless the user or the (user, item) is deleted."""
    owner = {}
    for g in range(len(groups) - 1, -1, -1):
        for x in groups[g]:
            owner[int(x)] = g
    gone, dels = set(map(tuple, pairs[:, :2].tolist())), set(del_user)
    out = [[] for _ in groups]
    for u, i, r in df[[0, 1, 2]].itertuples(index=False):
        if int(u) in owner and int(u) not in dels and (int(u), int(i)) not in gone:
            out[owner[int(u)]].append((float(u), float(i), r / max_rating))
    return [np.array(o, dtype=np.float64).reshape(-1, 3).T for o in out]


# ------------------------------------------------------------------------------------------------------------ CPU
def test_reference_pair_filter_equals_a_row_loop_and_the_draw_has_a_known_answer():
    df, n_user, del_user, pairs = _table(n=6000)
    groups = osisa.uniform_groups(n_user, 3)
    got, _ = _read_rating(df[0].values, df[1].values, df[2].values, n_user, 5, del_user, 3, groups, 'r',
                          del_rating=pairs)
    want = _brute(df, n_user, del_user, pairs, groups)
    for a, b in zip(got, want):
        assert a.shape == b.shape and np.array_equal(a, b)
    users, items = np.arange(10) + 100, np.arange(10) * 7
    d = _deletion_pairs(users, items, 20)
    assert d.dtype == np.int64 and d.tolist() == [[102, 14], [108, 56]]
    assert np.array_equal(d, np.stack([users, items], 1)[np.sort(np.random.RandomState(0).choice(10, 2, replace=False))])


@pytest.mark.parametrize("n_group", [1, 5, 7])
@pytest.mark.parametrize("sort", ['a', 'r'])
def test_host_read_rating_drops_deleted_pairs_like_the_oracle(n_group, sort):
    from ultrare_b200.read import readRating
    df, n_user, del_user, pairs = _table()
    got, gi = readRating(df, n_user, 5, del_user, pairs, n_group, [], sort)
    want, wi = _read_rating(df[0].values, df[1].values, df[2].values, n_user, 5, del_user, n_group, (), sort,
                            del_rating=pairs)
    assert [list(g) for g in gi] == [list(g) for g in wi]
    for a, b in zip(got, want):
        assert a.shape == b.shape and np.array_equal(a, b)
    # the group order is that of the unfiltered table
    _, gi0 = readRating(df, n_user, 5, [], [], n_group, [], sort)
    assert [list(g) for g in gi] == [list(g) for g in gi0]
    kept = sum(a.shape[1] for a in got)
    assert kept < sum(a.shape[1] for a in readRating(df, n_user, 5, del_user, [], n_group, [], sort)[0])


def test_negative_pair_ids_are_rejected_on_the_host():
    from ultrare_b200.read import readRating
    df, n_user, _, _ = _table(n=500)
    for bad in ([[-1, 3]], [[2, -4]]):
        with pytest.raises(ValueError):
            readRating(df, n_user, 5, [], bad, 2)


def _toy_env(tmp_path, monkeypatch):
    import ultrare_b200.config as cfg
    import ultrare_b200.group as grp
    from ultrare_b200 import synth
    data, save = str(tmp_path / "data"), str(tmp_path / "result")
    for mod in (cfg, grp):
        monkeypatch.setattr(mod, "DATA_DIR", data)
        monkeypatch.setattr(mod, "SAVE_DIR", save)
    synth.ensure_dataset("toy")
    return cfg, data, save


def test_inter_draw_and_cli(tmp_path, monkeypatch):
    cfg, _, _ = _toy_env(tmp_path, monkeypatch)
    p = cfg.InsParam("toy", 2, 1, [32], 3, 2, "inter")
    tr = pd.read_csv(p.train_dir, header=None)
    want = _deletion_pairs(tr[0].values, tr[1].values, 2)
    assert p.del_rating.dtype == np.int64 and np.array_equal(p.del_rating, want)
    assert len(want) == int(0.02 * len(tr)) and len(p.del_user) == 0
    assert len(cfg.InsParam("toy", 2, 1, [32], 3, 5, "inter").del_rating) == int(0.05 * len(tr))
    from ultrare_b200.main import _checked, parser
    assert _checked(parser.parse_args(['--deltype', 'inter', '--delper', '5'])).deltype == 'inter'
    with pytest.raises(AssertionError):
        _checked(parser.parse_args(['--deltype', 'core']))
    ins = cfg.Instance(p)
    assert ins.name == '/2/inter/toy_g3'
    saved = np.load(cfg.SAVE_DIR + ins.name + '/deletion.npy', allow_pickle=True)
    assert len(saved[0]) == 0 and np.array_equal(saved[1], want)


def test_instance_host_read_filters_training_only_and_routing_union(tmp_path, monkeypatch):
    cfg, _, _ = _toy_env(tmp_path, monkeypatch)
    monkeypatch.setenv("URE_HOST_INGEST", "1")
    ins = cfg.Instance(cfg.InsParam("toy", 2, 1, [32], 3, 2, "inter"))
    pairs = ins.param.del_rating
    train, idx, test, total = ins._read_data(True, 3, [])
    tr = pd.read_csv(ins.param.train_dir, header=None)
    te = pd.read_csv(ins.param.test_dir, header=None)
    want, widx = _read_rating(tr[0].values, tr[1].values, tr[2].values, ins.param.n_user, 5, (), 3, (), 'a',
                              del_rating=pairs)
    assert [list(g) for g in idx] == [list(g) for g in widx]
    for g in range(3):
        assert np.array_equal(train[g]._raw, want[g])
    assert sum(len(t) for t in train) == len(tr) - int(np.isin(tr[0].values * 2 ** 32 + tr[1].values,
                                                              pairs[:, 0] * 2 ** 32 + pairs[:, 1]).sum())
    test_want, _ = _read_rating(te[0].values, te[1].values, te[2].values, ins.param.n_user, 5, (), 3, idx, 'r')
    for g in range(3):
        assert np.array_equal(test[g]._raw, test_want[g])
    assert np.array_equal(total._raw, np.hstack(test_want))

    # routing: del_user, then the pair users it lacks, in first-appearance order (the loop it replaces)
    du = np.array([5, 9, 2], dtype=np.int64)
    assert cfg.routed_users(du, []) == list(du) and cfg.routed_users(du, np.zeros((0, 2), np.int64)) == list(du)
    loop = list(du)
    for rating in pairs:
        if rating[0] not in loop:
            loop.append(rating[0])
    assert cfg.routed_users(du, pairs) == loop
    assert cfg.routed_users([], pairs) == list(dict.fromkeys(pairs[:, 0].tolist()))


# ------------------------------------------------------------------------------------------------------------ GPU
def _device_equals_host(df, n_user, del_user, pairs, n_group, sort):
    import torch
    from ultrare_b200.read import RatingData, readRating, readRatingDevice
    host, gi_h = readRating(df, n_user, 5, del_user, pairs, n_group, [], sort)
    dev, gi_d, total = readRatingDevice(df, n_user, 5, del_user, pairs, n_group, [], sort, device='cuda')
    assert [list(g) for g in gi_h] == [list(g) for g in gi_d]
    row_of = torch.from_numpy(np.random.default_rng(1).integers(0, 50, n_user).astype(np.int32)).cuda()
    for g in range(n_group):
        want = RatingData(host[g])
        assert torch.equal(dev[g].records('cuda'), want.records('cuda')), g
        assert np.array_equal(dev[g]._raw, host[g])
        assert np.array_equal(dev[g].users, want.users) and np.array_equal(dev[g].items, want.items)
        assert np.array_equal(dev[g].ratings, want.ratings)
        assert torch.equal(dev[g].records_mapped('cuda', row_of, 't'), want.records_mapped('cuda', row_of, 't'))
    assert torch.equal(total.records('cuda'), RatingData(np.hstack(host)).records('cuda'))
    assert np.array_equal(total._raw, np.hstack(host))
    return host


@pytest.mark.gpu
@pytest.mark.parametrize("n_group,sort", [(1, 'r'), (5, 'a'), (7, 'r'), (7, 'a')])
def test_device_read_drops_deleted_pairs_like_the_host(cuda_dev, n_group, sort):
    df, n_user, del_user, pairs = _table(n=60000)
    _device_equals_host(df, n_user, del_user, pairs, n_group, sort)
    # one user with thousands of deleted items: the binary search over a long list
    rng = np.random.default_rng(3)
    heavy = pd.DataFrame({0: np.full(6000, 11), 1: rng.permutation(20000)[:6000], 2: rng.integers(1, 6, 6000)})
    big = pd.concat([df, heavy], ignore_index=True).sample(frac=1.0, random_state=4).reset_index(drop=True)
    hp = heavy.values[rng.choice(6000, 2500, replace=False)].astype(np.int64)
    host = _device_equals_host(big, n_user, [], np.concatenate([pairs, hp]), n_group, sort)
    kept = np.hstack(host)
    assert not np.isin(kept[0].astype(np.int64) * 2 ** 32 + kept[1].astype(np.int64), hp[:, 0] * 2 ** 32 + hp[:, 1]).any()


@pytest.mark.gpu
def test_device_pair_lists_both_layouts_and_rejections(cuda_dev):
    import torch
    from ultrare_b200 import kernels as kn
    from ultrare_b200.read import readRatingDevice
    t3 = torch.tensor([[0., 1., 5.], [1., 2., 4.], [0., 3., 1.], [1., 2., 2.], [0., 1., 3.]], dtype=torch.float64,
                      device='cuda')
    own = torch.tensor([1, 0], dtype=torch.int32, device='cuda')
    for pairs in (np.array([[0, 1], [1, 2], [0, 9], [5, 1]]), torch.tensor([[0, 1], [1, 2], [0, 9], [5, 1]], device='cuda')):
        lists = kn.deletion_lists(pairs, 2)
        assert lists[0].tolist() == [0, 2, 3] and lists[1].tolist() == [1, 9, 2]
        r_rows, o_rows = kn.partition_interactions(t3, 5, own, None, 2, columns=False, del_lists=lists)
        r_cols, o_cols = kn.partition_interactions(t3.t().contiguous(), 5, own, None, 2, columns=True, del_lists=lists)
        assert o_rows.tolist() == o_cols.tolist() == [0, 0, 1]            # rows past o[-1] are not written
        assert torch.equal(r_rows[:1], r_cols[:1]) and r_rows[:1, :2].tolist() == [[0, 3]]
    assert kn.deletion_lists(np.zeros((0, 2)), 2) is None and kn.deletion_lists([[7, 1]], 2) is None
    for bad in (np.array([[-1, 2]]), torch.tensor([[1, -2]], device='cuda')):
        with pytest.raises(ValueError):
            kn.deletion_lists(bad, 2)
    df, n_user, _, _ = _table(n=500)
    with pytest.raises(ValueError):
        readRatingDevice(df, n_user, 5, [], [[3, -1]], 2, device='cuda')


@pytest.mark.gpu
def test_device_pair_filter_at_20m_rows(cuda_dev):
    import torch
    from ultrare_b200 import kernels as kn
    rng = np.random.default_rng(11)
    n, n_user, n_item = 20_000_000, 138_493, 26_744
    u = np.sort(rng.integers(0, n_user, n))
    i = rng.integers(0, n_item, n)
    r = rng.integers(1, 6, n).astype(np.float64)
    rows = rng.choice(n, n // 100, replace=False)
    pairs = np.stack([u[rows], i[rows]], 1)
    table = kn.upload_table(np.stack([u.astype(np.float64), i.astype(np.float64), r]), cuda_dev)
    owner = torch.zeros(n_user, dtype=torch.int32, device=cuda_dev)
    rec, off = kn.partition_interactions(table, 5, owner, None, 1, del_lists=kn.deletion_lists(pairs, n_user))
    keys = u * 2 ** 32 + i
    keep = ~np.isin(keys, keys[rows])
    assert off.tolist() == [0, int(keep.sum())]
    got = rec[:int(keep.sum())].cpu().numpy()
    assert np.array_equal(got[:, 0], u[keep]) and np.array_equal(got[:, 1], i[keep])
    assert np.array_equal(got[:, 2].view(np.float32), (r[keep] / 5).astype(np.float32))


@pytest.mark.gpu
def test_sisa_unlearns_deleted_pairs_at_ml1m_shape(cuda_dev):
    """Pairs of shards 1 and 3 only: those two shards retrain on the device-filtered data, the others keep their
    tables bit for bit, no deleted pair is trained on, and the result equals unlearning on oracle-filtered arrays."""
    import torch
    from oracle import evalm as oev
    from ultrare_b200 import synth
    from ultrare_b200.method.sisa import Sisa
    from ultrare_b200.read import RatingData, loadData, readRating, readRatingDevice
    train, test = synth.ml_like()
    U, I, K, E, B = 6040, 3416, 5, 2, 30000
    tr = pd.DataFrame({0: train[0], 1: train[1], 2: train[2]})
    te = pd.DataFrame({0: test[0], 1: test[1], 2: test[2]})
    trr, groups = readRating(tr, U, 5, [], [], K, [], 'a')
    ter, _ = readRating(te, U, 5, [], [], K, groups)
    rng = np.random.default_rng(21)
    cand = np.flatnonzero(np.isin(train[0], np.concatenate([groups[1], groups[3]])))
    rows = rng.choice(cand, 4000, replace=False)
    pairs = np.stack([train[0][rows], train[1][rows]], 1).astype(np.int64)
    dev_tr, gi, _ = readRatingDevice(tr, U, 5, [], pairs, K, groups, 'r', device=cuda_dev)
    assert [list(g) for g in gi] == [list(g) for g in groups]
    ref_tr, _ = _read_rating(train[0], train[1], train[2], U, 5, (), K, groups, 'r', del_rating=pairs)

    class P:
        n_user, n_item, k, lam, seed, lr, lr_decay, momentum, epochs, batch = U, I, 16, 0.1, 42, 0.001, 0.95, 0.9, E, B

    test_dl = [loadData(RatingData(a), B, 1, False) for a in ter]
    test_total = np.hstack(ter)
    test_data = loadData(RatingData(test_total), B, 1, False)
    s1 = Sisa(P, 'mf', K, groups)
    s1.epoch_eval = 'none'
    before = s1.learn([loadData(RatingData(a), B, 1, True) for a in trr], test_dl, test_data, 0, '')
    w_before = before[0].user_mat.weight
    P_before = w_before.data.clone()
    Q_before = [m.item_mat.weight.data.clone() for m in before]
    del_user = sorted(set(pairs[:, 0].tolist()))

    keys = train[0].astype(np.int64) * 2 ** 32 + train[1].astype(np.int64)
    hit = np.isin(keys, pairs[:, 0] * 2 ** 32 + pairs[:, 1])
    assert sum(len(d) for d in dev_tr) == sum(a.shape[1] for a in trr) - int(hit.sum())
    gone = set(map(tuple, pairs.tolist()))
    for d in dev_tr:
        rec = d.records(cuda_dev).cpu().numpy()
        assert not gone & set(zip(rec[:, 0].tolist(), rec[:, 1].tolist()))

    def unlearn(datasets):
        for m in before:                       # every unlearn starts from the learnt tables
            m.user_mat.weight = w_before
        s = Sisa(P, 'mf', K, groups)
        s.epoch_eval = 'none'
        after = s.unlearn(before, [loadData(d, B, 1, True) for d in datasets], test_dl, test_data, del_user, 0, '')
        return s, after[0].user_mat.weight.data.clone(), [m.item_mat.weight.data.clone() for m in after]

    s2, P_after, Q_after = unlearn(dev_tr)
    assert s2.retrain_gid == set(osisa.route_deletions(groups, del_user)) == {1, 3}
    for g in range(K):
        rows_g = torch.as_tensor(np.asarray(groups[g]), device=P_after.device)
        if g in s2.retrain_gid:
            assert not torch.equal(Q_after[g], Q_before[g])
        else:
            assert torch.equal(Q_after[g], Q_before[g])
            assert torch.equal(P_after[rows_g], P_before[rows_g])
    final = dict(s2.final_log)

    s3, P_ref, Q_ref = unlearn([RatingData(a) for a in ref_tr])
    assert s3.retrain_gid == {1, 3}
    assert torch.equal(P_after, P_ref) and all(torch.equal(a, b) for a, b in zip(Q_after, Q_ref))

    tu, ti, trt = test_total[0].astype(np.int64), test_total[1].astype(np.int64), test_total[2].astype(np.float32)
    rmse, ndcg, hr, _ = oev.base_test([P_after.cpu().numpy()] * K, [q.cpu().numpy() for q in Q_after], tu, ti, trt)
    assert abs(final['total_rmse'] - rmse) < 1e-4 * rmse
    assert abs(final['total_ndcg'] - ndcg) < 1e-4 and abs(final['total_hr'] - hr) < 1e-4


@pytest.mark.gpu
def test_cli_deltype_inter_end_to_end(cuda_dev, tmp_path, monkeypatch):
    cfg, _, save = _toy_env(tmp_path, monkeypatch)
    from ultrare_b200.main import main
    common = ['--dataset', 'toy', '--synth', '--deltype', 'inter', '--epoch', '2', '--worker', '1', '--verbose', '0']
    main(common + ['--group', '0'])
    assert os.path.exists(save + '/2/inter/toy_g0/MF_full_train/user_mat0.npy')
    assert os.path.exists(save + '/2/inter/toy_g0/MF_retrain/user_mat0.npy')
    ins = main(common + ['--group', '3', '--recommend', '10'])
    gdir = save + '/2/inter/toy_g3'
    for sub in ('MF_emb-ot_sisa_learn', 'MF_emb-ot_sisa_unlearn'):
        assert os.path.exists(f'{gdir}/{sub}/rec10.npy'), sub
    tr = pd.read_csv(ins.param.train_dir, header=None)
    pairs = _deletion_pairs(tr[0].values, tr[1].values, 2)
    saved = np.load(gdir + '/deletion.npy', allow_pickle=True)
    assert np.array_equal(saved[1], pairs) and len(saved[0]) == 0
    sisa = ins.last_sisa
    assert sisa.retrain_gid == osisa.route_deletions(sisa.group_index, pairs[:, 0])
    filt, _ = _read_rating(tr[0].values, tr[1].values, tr[2].values, ins.param.n_user, 5, (), 1, (), 'r',
                           del_rating=pairs)
    rec = np.load(gdir + '/MF_emb-ot_sisa_unlearn/rec10.npy')
    seen = {}
    for u, i in zip(filt[0][0].astype(np.int64), filt[0][1].astype(np.int64)):
        seen.setdefault(int(u), set()).add(int(i))
    for u in range(rec.shape[0]):
        assert not seen.get(u, set()) & set(rec[u].tolist()), u
