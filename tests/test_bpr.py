"""BPR training of the shard models (ure_mf_train_bpr, ShardBatch(loss='bpr'), Sisa / Scratch with loss='bpr', the
--loss flag) against the fp32 NumPy restatement in oracle/bpr.py."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle import bpr as obpr, mf as omf, sisa as osisa

K_TOY = 3


# ------------------------------------------------------------------------------------------------------------ fixtures
def _toy_source(tmp_path, K=K_TOY):
    """The toy data as CSV files and the source dict of a Sisa learned from them (uniform grouping)."""
    import pandas as pd
    z = np.load(os.path.join(ROOT, "tests", "golden", "toy_data.npz"))
    paths = {}
    for part in ("train", "test"):
        p = str(tmp_path / f"toy_{part}.csv")
        pd.DataFrame({0: z[part + "_u"].astype(np.int64), 1: z[part + "_i"].astype(np.int64),
                      2: z[part + "_r2"] / 2.0}).to_csv(p, header=False, index=False)
        paths[part] = p
    return dict(dataset='toy', train_file=paths["train"], test_file=paths["test"], max_rating=5, grouping='uniform',
                group_index=osisa.uniform_groups(1508, K))


def _manifest(tmp_path, src, **over):
    from ultrare_b200.method import sisa_state as st
    size, sha = st.file_digest(src['train_file'])
    man = dict(format=st.FORMAT_VERSION, K=K_TOY, slices=1, k=16, n_user=1508, n_item=2071, epochs=2, batch=3000,
               lr=0.001, lr_decay=0.95, lam=0.1, momentum=0.9, seed=42, combine='mean', epoch_eval='final',
               dataset='toy', grouping='uniform', max_rating=5,
               train_file=dict(path=src['train_file'], bytes=size, sha256=sha), test_file=src['test_file'], requests=0)
    man.update(over)
    d = tmp_path / "state"
    d.mkdir(exist_ok=True)
    (d / "manifest.json").write_text(json.dumps(man))
    return str(d), man


def _heavy_set(n_user=40, n_item=300, seed=5):
    """Records with a user holding >= 60 % of the catalogue, one holding all of it, and light users."""
    rng = np.random.default_rng(seed)
    u, i = [], []
    for x in range(n_user):
        if x == 0:
            items = np.arange(n_item)                                   # the whole catalogue: every triple dropped
        elif x == 1:
            items = rng.choice(n_item, int(0.65 * n_item), replace=False)
        else:
            items = rng.choice(n_item, int(rng.integers(1, 30)), replace=False)
        u += [x] * len(items)
        i += list(items)
    perm = rng.permutation(len(u))
    return np.asarray(u, np.int64)[perm], np.asarray(i, np.int64)[perm], n_user, n_item


# ------------------------------------------------------------------------------------------------------------ CPU
def test_oracle_sampler_never_returns_a_seen_item_and_is_deterministic():
    u, i, _, n_item = _heavy_set()
    seen = set(zip(u.tolist(), i.tolist()))
    for ep in range(3):
        neg = obpr.negatives(u, i, n_item, 42, 2, ep)
        assert np.array_equal(neg, obpr.negatives(u, i, n_item, 42, 2, ep))
        ok = neg >= 0
        assert ok.sum() > 0.9 * (u != 0).sum()
        assert all((a, b) not in seen for a, b in zip(u[ok].tolist(), neg[ok].tolist()))
        assert ((neg >= -1) & (neg < n_item)).all()
    assert not np.array_equal(obpr.negatives(u, i, n_item, 42, 2, 0), obpr.negatives(u, i, n_item, 42, 2, 1))


def test_oracle_sampler_drops_users_whose_candidates_are_all_seen():
    u, i, _, n_item = _heavy_set()
    neg = obpr.negatives(u, i, n_item, 42, 0, 0)
    assert (neg[u == 0] == -1).all()                                   # rated every item
    # a constructed user: its only record's 16 candidates are exactly its other records' items
    n_item = 1000
    c = obpr.candidates(omf.perm_key(7, 1, 0), 1, n_item)[0].astype(np.int64)
    items = np.unique(np.concatenate([[c[0]], c]))
    uu = np.zeros(len(items), np.int64)
    ii = np.concatenate([[c[0]], np.setdiff1d(items, [c[0]])])          # record 0 holds item c_0 itself
    got, tries = obpr.negatives(uu, ii, n_item, 7, 1, 0, return_tries=True)
    assert got[0] == -1 and tries[0] == obpr.CANDIDATES


def test_oracle_sampler_is_roughly_uniform_over_unseen_items():
    from scipy import stats
    rng = np.random.default_rng(0)
    n_item, n = 50, 40000
    u = np.zeros(n, np.int64)
    i = rng.integers(0, 10, n)                                         # the user has seen items 0..9
    neg = obpr.negatives(u, i, n_item, 3, 0, 0)
    assert (neg >= 10).all()
    counts = np.bincount(neg, minlength=n_item)[10:]
    assert stats.chisquare(counts).pvalue > 1e-4


def test_bpr_refuses_schedules_other_than_dense():
    from ultrare_b200 import kernels as kn
    assert kn._bpr_mode("bpr", None) == "dense" and kn._bpr_mode("bpr", "auto") == "dense"
    assert kn._bpr_mode("mse", "owner") == "owner"
    for mode in ("owner", "lazy", "runs"):
        with pytest.raises(ValueError, match="dense"):
            kn._bpr_mode("bpr", mode)
    with pytest.raises(ValueError, match="loss"):
        kn._bpr_mode("hinge", None)


def test_cli_refuses_bpr_with_the_fitted_combination():
    from ultrare_b200.main import _checked, parser
    with pytest.raises(AssertionError, match="--combine fit"):
        _checked(parser.parse_args(['--loss', 'bpr', '--combine', 'fit']))
    assert _checked(parser.parse_args(['--loss', 'bpr'])).loss == 'bpr'
    assert _checked(parser.parse_args([])).loss == 'mse'


def test_request_run_with_a_conflicting_loss_is_refused(tmp_path):
    from ultrare_b200.main import main
    src = _toy_source(tmp_path)
    d, _ = _manifest(tmp_path, src, loss='bpr')
    (tmp_path / "u.txt").write_text("3\n")
    req = ['--unlearn-from', d, '--out', str(tmp_path / "out"), '--forget-users', str(tmp_path / "u.txt")]
    with pytest.raises(AssertionError, match="--loss"):
        main(req + ['--loss', 'mse'])


def test_manifest_without_loss_reads_as_mse(tmp_path):
    from ultrare_b200.method import sisa_state as st
    src = _toy_source(tmp_path)
    d, man = _manifest(tmp_path, src)
    assert 'loss' not in man and st.read_manifest(d)['loss'] == 'mse'
    d, _ = _manifest(tmp_path, src, loss='bpr')
    assert st.read_manifest(d)['loss'] == 'bpr'
    d, _ = _manifest(tmp_path, src, loss='hinge')
    with pytest.raises(ValueError, match="loss"):
        st.read_manifest(d)


# ------------------------------------------------------------------------------------------------------------ GPU
def _torch():
    import torch
    return torch


@pytest.mark.gpu
def test_device_negatives_equal_the_oracle_on_toy(toy, cuda_dev):
    from ultrare_b200 import kernels as kn
    u, i, r = toy["train"]
    inter = kn.pack_interactions(u, i, r / 5.0, cuda_dev)
    seen = kn.seen_lists(inter, toy["n_user"], toy["n_item"])
    for sid, ep in ((0, 0), (3, 7)):
        got, tries = kn.bpr_negatives(inter, toy["n_item"], seen, 42, sid, ep, want_tries=True)
        want, wt = obpr.negatives(u, i, toy["n_item"], 42, sid, ep, return_tries=True)
        assert np.array_equal(got.cpu().numpy(), want) and np.array_equal(tries.cpu().numpy(), wt)


@pytest.mark.gpu
@pytest.mark.parametrize("table", ["compact", "full"])
def test_device_negatives_equal_the_oracle_with_heavy_users(cuda_dev, table):
    """A user with >= 60 % of the catalogue (several candidates each) and one with all of it (dropped); compact user
    table = rows 0..n-1 of the shard's users, full = global ids in a larger table."""
    from ultrare_b200 import kernels as kn
    u, i, n_user, n_item = _heavy_set()
    if table == "full":
        u = u * 7 + 3
        n_user = int(u.max()) + 20
    inter = kn.pack_interactions(u, i, np.ones(len(u)), cuda_dev)
    seen = kn.seen_lists(inter, n_user, n_item)
    for ep in range(3):
        got = kn.bpr_negatives(inter, n_item, seen, 11, 4, ep).cpu().numpy()
        assert np.array_equal(got, obpr.negatives(u, i, n_item, 11, 4, ep))
    assert (got[u == u.min()] == -1).all() if table == "compact" else True


def _bpr_shards(dev, K, d, epochs, batch, explicit, n_user=300, n_item=200, seed=0, sizes=None):
    torch = _torch()
    from ultrare_b200 import kernels as kn
    rng = np.random.default_rng(seed)
    shards, host = [], []
    for s in range(K):
        n = sizes[s] if sizes else int(rng.integers(2500, 4000))
        u, i = rng.integers(0, n_user, n), rng.integers(0, n_item, n)
        P0 = (rng.standard_normal((n_user, d)) * 0.3).astype(np.float32)
        Q0 = (rng.standard_normal((n_item, d)) * 0.3).astype(np.float32)
        perms = [omf.feistel_perm(n, omf.perm_key(9, s + 1, ep)) for ep in range(epochs)]
        perm_t = torch.tensor(np.stack(perms).astype(np.int32), device=dev) if explicit else None
        shards.append(kn.ShardState(kn.pack_interactions(u, i, np.ones(n), dev), torch.tensor(P0, device=dev),
                                    torch.tensor(Q0, device=dev), epochs, shard_id=s + 1, perm_seed=9, perm=perm_t))
        host.append((u, i, P0, Q0, perms))
    return shards, host


@pytest.mark.gpu
@pytest.mark.parametrize("d,K,explicit", [(8, 1, True), (16, 3, False), (32, 5, True), (64, 3, False),
                                          (128, 1, False), (16, 5, True)])
def test_bpr_training_equals_the_oracle(cuda_dev, d, K, explicit):
    """K shards in one launch, ragged last batch: weights 1e-4 abs, losses 1e-3 rel over 3 epochs."""
    from ultrare_b200 import kernels as kn
    epochs, batch = 3, 1000
    shards, host = _bpr_shards(cuda_dev, K, d, epochs, batch, explicit, seed=d + K)
    assert any(s.n % batch for s in shards)
    sb = kn.ShardBatch(shards, d, batch, loss="bpr")
    assert sb.mode == "dense"
    sb.train()
    losses = sb.train_losses()
    for s in range(K):
        u, i, P0, Q0, perms = host[s]
        P, Q, _, _, ls = obpr.bpr_train(P0, Q0, u, i, perms, batch, epochs, 9, s + 1)
        np.testing.assert_allclose(losses[s], ls, rtol=1e-3)
        assert np.abs(shards[s].P.cpu().numpy() - P).max() < 1e-4
        assert np.abs(shards[s].Q.cpu().numpy() - Q).max() < 1e-4


@pytest.mark.gpu
def test_bpr_training_across_the_steplr_boundary(cuda_dev):
    """70 epochs, 20 of them after StepLR's decay at epoch 50.  Two device runs differ only by the order of the float
    atomics; the oracle must lie within 20x their spread, floored at 2e-5.  The same oracle without the decay lies
    1.2e-2 away, so a kernel that skipped or misplaced the decay fails by a factor of several hundred."""
    from ultrare_b200 import kernels as kn
    epochs, batch, d = 70, 500, 16
    runs = []
    for _ in range(2):
        shards, host = _bpr_shards(cuda_dev, 1, d, epochs, batch, False, seed=77, sizes=[3500])
        sb = kn.ShardBatch(shards, d, batch, loss="bpr")
        sb.train()
        runs.append((shards[0].P.cpu().numpy(), shards[0].Q.cpu().numpy(), sb.train_losses()[0]))
    u, i, P0, Q0, perms = host[0]
    P, Q, _, _, ls = obpr.bpr_train(P0, Q0, u, i, perms, batch, epochs, 9, 1)
    Pn, Qn, _, _, _ = obpr.bpr_train(P0, Q0, u, i, perms, batch, epochs, 9, 1, lr_decay=1.0)
    spread = max(np.abs(runs[0][0] - runs[1][0]).max(), np.abs(runs[0][1] - runs[1][1]).max())
    err = max(np.abs(runs[0][0] - P).max(), np.abs(runs[0][1] - Q).max())
    bound = max(2e-5, 20 * spread)
    print(f"steplr: device spread {spread:.3g}, oracle error {err:.3g}, bound {bound:.3g}")
    assert err <= bound
    assert max(np.abs(runs[0][0] - Pn).max(), np.abs(runs[0][1] - Qn).max()) > 100 * bound
    np.testing.assert_allclose(runs[0][2], ls, rtol=1e-3)


@pytest.mark.gpu
def test_bpr_epoch_by_epoch_equals_one_launch(cuda_dev):
    from ultrare_b200 import kernels as kn
    a, _ = _bpr_shards(cuda_dev, 3, 16, 3, 1000, False, seed=3)
    b, _ = _bpr_shards(cuda_dev, 3, 16, 3, 1000, False, seed=3)
    sa, sb = kn.ShardBatch(a, 16, 1000, loss="bpr"), kn.ShardBatch(b, 16, 1000, loss="bpr")
    sa.train()
    for t in range(1, sb.total_steps + 1):
        sb.train(t)
    for x, y in zip(a, b):
        assert np.abs(x.P.cpu().numpy() - y.P.cpu().numpy()).max() < 1e-4
        assert np.abs(x.Q.cpu().numpy() - y.Q.cpu().numpy()).max() < 1e-4
    for la, lb in zip(sa.train_losses(), sb.train_losses()):
        np.testing.assert_allclose(la, lb, rtol=1e-5)


# ---- Sisa with BPR
class _Param:
    def __init__(self, epochs, loss='bpr'):
        self.n_user, self.n_item, self.k, self.lam = 1508, 2071, 16, 0.1
        self.seed, self.lr, self.lr_decay, self.momentum = 42, 0.001, 0.95, 0.9
        self.epochs, self.batch, self.loss = epochs, 3000, loss


def _read(src, R, users=(), pairs=()):
    from ultrare_b200.method import sisa_state as st
    return st.read_retained(src, 1508, K_TOY, R, 3000, np.asarray(users, dtype=np.int64),
                            np.asarray(pairs, dtype=np.int64).reshape(-1, 2))


def _sisa(src, idx, R, E=2):
    from ultrare_b200.method.sisa import Sisa
    s = Sisa(_Param(E), 'mf', len(idx), idx)
    s.epoch_eval, s.slices, s.source = 'final', R, dict(src)
    return s


def _tables(s):
    return (s.model_list[0].user_mat.weight.data.cpu().numpy().copy(),
            [m.item_mat.weight.data.cpu().numpy().copy() for m in s.model_list])


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 4])
@pytest.mark.parametrize("kind", ["users", "pairs"])
def test_sisa_bpr_unlearn_retrains_only_affected_shards(cuda_dev, tmp_path, R, kind):
    """learn -> unlearn: shards the request does not touch keep their tables bit for bit; every shard is within the
    training tolerance of a BPR learn on the retained data (R = 4: from the stored checkpoint of its first affected
    slice, which stays as it was)."""
    src = _toy_source(tmp_path)
    tl, sl, total, idx = _read(src, R)
    s = _sisa(src, idx, R)
    s.learn(tl, sl, total, 0, '')
    P0, Q0 = _tables(s)
    ck0 = {g: [(a.cpu().numpy().copy(), b.cpu().numpy().copy()) for a, b in getattr(m, 'checkpoints', [])]
           for g, m in enumerate(s.model_list)}
    g0 = idx[0]
    if kind == "users":
        users, pairs = [g0[len(g0) - 3], g0[len(g0) - 1]], []
    else:
        u, i, _ = np.loadtxt(src['train_file'], delimiter=',', unpack=True)
        row = np.flatnonzero(u == g0[-2])[0]
        users, pairs = [], [[int(u[row]), int(i[row])]]
    from ultrare_b200.config import routed_users
    tl2, sl2, total2, _ = _read(src, R, users, pairs)
    s.unlearn(list(s.model_list), tl2, sl2, total2, routed_users(users, np.asarray(pairs).reshape(-1, 2)), 0, '')
    P1, Q1 = _tables(s)
    for g in (1, 2):
        assert np.array_equal(Q1[g], Q0[g]), g
        rows = np.asarray(idx[g])
        assert np.array_equal(P1[rows], P0[rows]), g
    if R > 1:
        first = int(s.first_slice[0])
        ck1 = [(a.cpu().numpy(), b.cpu().numpy()) for a, b in s.model_list[0].checkpoints]
        for r in range(first + 1):
            assert np.array_equal(ck1[r][0], ck0[0][r][0]) and np.array_equal(ck1[r][1], ck0[0][r][1]), r
    if R > 1:                   # a sliced learn on the retained data draws the same initial weights
        ref = _sisa(src, idx, R)
        ref.learn(tl2, sl2, total2, 0, '')
        Pr, Qr = _tables(ref)
        for g in range(K_TOY):
            assert np.abs(Q1[g] - Qr[g]).max() < 1e-4, g
        keep = np.setdiff1d(np.arange(1508), users)
        assert np.abs(P1[keep] - Pr[keep]).max() < 1e-4
    else:                       # unsliced: shard 0 retrains alone from the draw of its own generator -- a BPR learn of
        import torch            # that one shard on the retained data with the same seed
        from ultrare_b200 import kernels as kn
        from ultrare_b200.method.scratch import model_generator
        rec = tl2[0].dataset.records_mapped(cuda_dev, s._row_of, 'sisa_local')
        sb = kn.ArenaShardBatch([rec], [len(idx[0])], 2071, 16, 3000, 2, [1], 42,
                                generator=lambda: model_generator(42, 1, cuda_dev), loss='bpr')
        sb.train()
        torch.cuda.synchronize()
        v = sb.shards[0]
        assert np.abs(Q1[0] - v.Q.cpu().numpy()).max() < 1e-4
        keep = np.setdiff1d(np.asarray(idx[0]), users)
        assert np.abs(P1[keep] - v.P.cpu().numpy()[s._row_of_np[keep]]).max() < 1e-4


def _local(s):
    """The merged user table and this rank's item tables."""
    return (s.model_list[0].user_mat.weight.data.cpu().numpy().copy(),
            {g: m.item_mat.weight.data.cpu().numpy().copy() for g, m in enumerate(s.model_list)
             if getattr(m, 'item_mat', None) is not None})


@pytest.mark.gpu
def test_sisa_bpr_two_ranks_equal_one_gpu(cuda_dev, tmp_path, monkeypatch):
    """Learn and unlearn at 2 ranks (threads on one GPU, each training its own shards against seen lists of its own
    records) agree with one GPU within the training tolerance: merged user table and every rank's item tables.  The
    weights are drawn per shard on the host (init_on_device = False), so both worlds start from the same tables."""
    from test_sisa_state import _Ranks
    src = _toy_source(tmp_path)
    tl, sl, total, idx = _read(src, 1)
    users = [idx[0][3], idx[1][7], idx[2][11]]
    tl2, sl2, total2, _ = _read(src, 1, users)

    def run(dist=None):
        s = _sisa(src, idx, 1)
        s.init_on_device = False
        if dist is not None:
            s.dist = dist
        s.learn(tl, sl, total, 0, '')
        learned = _local(s)
        s.unlearn(list(s.model_list), tl2, sl2, total2, users, 0, '')
        return learned, _local(s)

    one = run()
    ranks = _Ranks(2)
    ranks.serialise(monkeypatch, _sisa(src, idx, 1))
    got = ranks.run(lambda r: run(ranks.dist(r)))
    seen = set()
    for r, per_rank in enumerate(got):
        for (P, Q), (P1, Q1) in zip(per_rank, one):
            assert np.abs(P - P1).max() < 1e-4, r
            for g, q in Q.items():
                assert g % 2 == r and np.abs(q - Q1[g]).max() < 1e-4, (r, g)
                seen.add(g)
    assert seen == set(range(K_TOY))


@pytest.mark.gpu
def test_sisa_bpr_faithful_full_tables_equal_the_oracle(cuda_dev, tmp_path):
    """epoch_eval='faithful' trains full (global-id) user tables: with injected initial weights every shard equals the
    BPR oracle on its records, the seen lists indexed by global user id."""
    from ultrare_b200.method.sisa import Sisa
    from ultrare_b200.method.utils import MF
    from conftest import init_weights

    class Injected(Sisa):
        def _new_model(self, id, user_rows=None):
            assert user_rows is None
            return MF.from_weights(*init_weights(200 + id))

    src = _toy_source(tmp_path)
    tl, sl, total, idx = _read(src, 1)
    s = Injected(_Param(2), 'mf', K_TOY, idx)
    s.epoch_eval, s.slices, s.source = 'faithful', 1, dict(src)
    s.learn(tl, sl, total, 0, '')
    for g in range(K_TOY):
        rec = tl[g].dataset.records(cuda_dev).cpu().numpy()
        u, i = rec[:, 0].astype(np.int64), rec[:, 1].astype(np.int64)
        perms = [omf.feistel_perm(len(u), omf.perm_key(42, g + 1, ep)) for ep in range(2)]
        P0, Q0 = init_weights(201 + g)
        P, Q, _, _, _ = obpr.bpr_train(P0, Q0, u, i, perms, 3000, 2, 42, g + 1)
        m = s.model_list[g]
        assert m.user_mat.weight.shape[0] == 1508
        rows = np.asarray(idx[g])
        assert np.abs(m.item_mat.weight.data.cpu().numpy() - Q).max() < 1e-4, g
        assert np.abs(s.model_list[0].user_mat.weight.data.cpu().numpy()[rows] - P[rows]).max() < 1e-4, g


@pytest.mark.gpu
def test_sisa_bpr_recommend_and_state_round_trip(cuda_dev, tmp_path):
    """recommend returns valid lists without seen items; save -> load is bit-equal; a request from the loaded state is
    within the training tolerance of the in-process unlearn."""
    from ultrare_b200.method.sisa import Sisa
    src = _toy_source(tmp_path)
    tl, sl, total, idx = _read(src, 1)
    s = _sisa(src, idx, 1)
    s.learn(tl, sl, total, 0, '')
    items, scores = s.recommend(None, 10, exclude=tl)
    items = items.cpu().numpy()
    u, i, _ = np.loadtxt(src['train_file'], delimiter=',', unpack=True)
    seen = set(zip(u.astype(int).tolist(), i.astype(int).tolist()))
    assert ((items >= 0) & (items < 2071)).all()
    assert all((x, int(it)) not in seen for x in range(0, 1508, 37) for it in items[x])
    s.save_state(str(tmp_path / "st"))
    s._join_writers()
    man = json.loads((tmp_path / "st" / "manifest.json").read_text())
    assert man['loss'] == 'bpr'
    L = Sisa.load_state(str(tmp_path / "st"))
    assert L.loss == 'bpr'
    Pa, Qa = _tables(s)
    Pb, Qb = _tables(L)
    assert np.array_equal(Pa, Pb) and all(np.array_equal(a, b) for a, b in zip(Qa, Qb))
    users = [idx[1][0], idx[1][5]]
    tl2, sl2, total2 = L.retained_data(users, ())
    L.apply_request(users, (), tl2, sl2, total2, 0, '')
    s.unlearn(list(s.model_list), tl2, sl2, total2, users, 0, '')
    Pa, Qa = _tables(s)
    Pb, Qb = _tables(L)
    assert np.abs(Pa - Pb).max() < 1e-4 and max(np.abs(a - b).max() for a, b in zip(Qa, Qb)) < 1e-4


@pytest.mark.gpu
def test_sisa_bpr_refuses_the_fitted_combination(cuda_dev, tmp_path):
    src = _toy_source(tmp_path)
    tl, sl, total, idx = _read(src, 1)
    s = _sisa(src, idx, 1)
    s.combine = 'fit'
    with pytest.raises(ValueError, match="BPR"):
        s.learn(tl, sl, total, 0, '')


# ---- CLI end to end
def _main(env, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "main.py"), *args], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return r.stdout


@pytest.mark.gpu
def test_cli_bpr_runs_end_to_end(cuda_dev, tmp_path):
    env = dict(os.environ, ULTRARE_ROOT=str(tmp_path))
    _main(env, "--dataset", "toy", "--synth", "--group", "0", "--loss", "bpr", "--epoch", "2", "--verbose", "0")
    full = tmp_path / "result" / "2" / "rand" / "toy_g0_bpr" / "MF_full_train"
    assert (full / "user_mat0.npy").exists()
    assert not (tmp_path / "result" / "2" / "rand" / "toy_g0").exists()      # never the MSE run's directory
    _main(env, "--dataset", "toy", "--synth", "--group", "3", "--loss", "bpr", "--grouping", "rating-ot", "--slices",
          "2", "--recommend", "10", "--save-state", "--epoch", "2", "--verbose", "0")
    gdir = tmp_path / "result" / "2" / "rand" / "toy_g3_bpr"
    learn = gdir / "MF_rating-ot_sisa_learn"
    assert (learn / "rec10.npy").exists()
    assert json.loads((learn / "state" / "manifest.json").read_text())['loss'] == 'bpr'
    u, i = np.loadtxt(tmp_path / "data" / "toy" / "0_train.csv", delimiter=',', usecols=(0, 1), unpack=True,
                      max_rows=2)
    (tmp_path / "r.csv").write_text(f"{int(u[0])},{int(i[0])}\n{int(u[1])},{int(i[1])}\n")
    out = tmp_path / "req"
    _main(env, "--unlearn-from", str(learn / "state"), "--out", str(out), "--forget-ratings", str(tmp_path / "r.csv"),
          "--verbose", "0", "--recommend", "10")
    assert json.loads((out / "state" / "manifest.json").read_text())['loss'] == 'bpr'
    assert (out / "rec10.npy").exists() and (out / "slices.npy").exists()
