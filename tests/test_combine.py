"""Learned combination of the SISA shard models: the float64 oracle (oracle/combine.py) against least squares on the
augmented system and the --combine flag (CPU); the Gram, weighted-sum and group-score kernels against float64, Sisa
with combine='fit' against the oracle fitted on the retained rows, several ranks against one GPU, and the CLI end to
end with interaction-level deletions (GPU)."""
import os
import threading

import numpy as np
import pandas as pd
import pytest

from conftest import load_gold
from oracle import combine as ocomb
from oracle import recommend as orec
from oracle import sisa as osisa

D_ALL = (8, 16, 32, 64, 128)


def _gram_row(G, m, n, K):
    """The kernel's layout of one group: upper triangle of G row by row, the moments, the row count."""
    return np.concatenate([G[np.triu_indices(K + 1)], m, [n]])


# ------------------------------------------------------------------------------ CPU
def test_oracle_solve_is_least_squares_on_the_augmented_system_and_the_product_solve_agrees():
    """The ridge solve with a free intercept == np.linalg.lstsq of [X 1; sqrt(lambda) I 0] [w; b] = [r; 0]; the
    product's solve_combination on the kernel layout of the same Gram gives the same weights; an empty group and a
    user in no group get the mean combination."""
    from ultrare_b200.method.utils import solve_combination
    rng = np.random.default_rng(0)
    for K, n in ((1, 7), (3, 40), (5, 500), (8, 2000)):
        X = rng.standard_normal((n, K)) * rng.uniform(0.1, 3.0, K) + rng.standard_normal(K)
        r = X @ rng.standard_normal(K) + 0.3 + 0.1 * rng.standard_normal(n)
        G, m, cnt = ocomb.gram(X, r)
        w, b = ocomb.solve(G, m, cnt, K)
        lam = ocomb.RIDGE * np.trace(G[:K, :K]) / K
        A = np.block([[X, np.ones((n, 1))], [np.sqrt(lam) * np.eye(K), np.zeros((K, 1))]])
        ref = np.linalg.lstsq(A, np.concatenate([r, np.zeros(K)]), rcond=None)[0]
        np.testing.assert_allclose(np.append(w, b), ref, rtol=1e-8, atol=1e-10)
        pw, pb = solve_combination(np.stack([_gram_row(G, m, cnt, K), np.zeros(len(_gram_row(G, m, cnt, K)))]), K)
        np.testing.assert_allclose(pw[0], w, rtol=1e-10, atol=1e-12)
        assert pb[0] == pytest.approx(b, rel=1e-10, abs=1e-12)
        np.testing.assert_array_equal(pw[1], np.full(K, 1.0 / K))        # no rows: the mean
        assert pb[1] == 0.0
    w, b = ocomb.solve(np.zeros((4, 4)), np.zeros(4), 0, 3)
    assert np.array_equal(w, np.full(3, 1 / 3)) and b == 0.0
    P = rng.standard_normal((4, 8))
    Qs = [rng.standard_normal((5, 8)) for _ in range(3)]
    owner = np.array([0, -1, 2, 1])
    W, B = rng.standard_normal((3, 3)), rng.standard_normal(3)
    s = ocomb.scores(P, Qs, W, B, owner, [1, 2], [4, 0])
    assert s[0] == pytest.approx(np.mean([P[1] @ Q[4] for Q in Qs]))          # user 1 is in no group
    assert s[1] == pytest.approx(B[2] + sum(W[2, k] * (P[2] @ Qs[k][0]) for k in range(3)))


def test_combine_flag_parses_and_defaults_to_the_mean():
    from ultrare_b200.config import Instance
    from ultrare_b200.main import _checked, parser
    assert vars(parser.parse_args([]))['combine'] == 'mean' and Instance.combine == 'mean'
    assert _checked(parser.parse_args(['--combine', 'fit'])).combine == 'fit'
    with pytest.raises(SystemExit):
        parser.parse_args(['--combine', 'attention'])


def test_sisa_rejects_an_unknown_combine_and_a_missing_fit():
    """Sisa.combine other than 'mean' / 'fit' raises ValueError; 'fit' without a fitted combination raises a
    RuntimeError that says so (no CUDA device needed: the checks run before any kernel)."""
    from ultrare_b200.method.sisa import Sisa
    s = Sisa.__new__(Sisa)
    s.combine, s.combination = 'mean', None
    assert s._use_fit() is False
    s.combine = 'attention'
    with pytest.raises(ValueError, match="'mean' or 'fit'"):
        s._use_fit()
    s.combine = 'fit'
    assert s._use_fit() is True
    with pytest.raises(RuntimeError, match="no combination has been fitted"):
        s._fitted()


# ------------------------------------------------------------------------------ GPU helpers
def _dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _records(rng, n_user, n_item, n, dev):
    import torch
    r = np.zeros((n, 4), dtype=np.int32)
    r[:, 0] = rng.integers(0, n_user, n)
    r[:, 1] = rng.integers(0, n_item, n)
    r[:, 2] = (rng.integers(1, 6, n).astype(np.float32) / 5).view(np.int32)
    return torch.from_numpy(r).to(dev)


def _oracle_gram(P, Qs, rec, K):
    """float64 Gram of z = [x; 1; r] over the records, computed on the device from the same fp32 tables, in the
    kernel's layout, and the diagonal scale sqrt(G_aa G_bb) of every entry."""
    import torch
    u, i = rec[:, 0].long(), rec[:, 1].long()
    r = rec[:, 2].view(torch.float32).double()
    P64 = P.double()[u]
    cols = [(P64 * Q.double()[i]).sum(1) for Q in Qs]
    Z = torch.stack(cols + [torch.ones_like(r), r], 1)
    F = (Z.T @ Z).cpu().numpy()
    a, b = np.triu_indices(K + 1)
    a = np.concatenate([a, np.arange(K + 1), [K]])
    b = np.concatenate([b, np.full(K + 1, K + 1), [K]])
    diag = np.diag(F)
    return F[a, b], np.sqrt(diag[a] * diag[b])


def _check_gram(got, P, Qs, rec, K):
    want, scale = _oracle_gram(P, Qs, rec, K)
    assert got[-1] == rec.shape[0]
    assert np.all(np.abs(got - want) <= 1e-5 * scale), np.max(np.abs(got - want) / np.maximum(scale, 1e-300))


# ------------------------------------------------------------------------------ GPU: kernels
@pytest.mark.gpu
@pytest.mark.parametrize("d", D_ALL)
def test_gram_kernel_vs_float64(d):
    """Every d, K in {1, 2, 5, 8, 64}, groups of 0, 1, 31, 32, 33 and 10^6 + 7 rows in one call; entry-wise error
    <= 1e-5 sqrt(G_aa G_bb); two calls bit-identical."""
    import torch
    from ultrare_b200 import kernels as kn
    dev = _dev()
    rng = np.random.default_rng(d)
    n_user, n_item = 5000, 3000
    P = torch.from_numpy(rng.standard_normal((n_user, d), dtype=np.float32)).to(dev)
    for K in (1, 2, 5, 8, 64):
        Qs = [torch.from_numpy(rng.standard_normal((n_item, d), dtype=np.float32)).to(dev) for _ in range(K)]
        recs = [_records(rng, n_user, n_item, n, dev) for n in (0, 1, 31, 32, 33, 1_000_007)]
        a = kn.combine_gram(P, Qs, recs).cpu().numpy()
        b = kn.combine_gram(P, Qs, recs).cpu().numpy()
        assert a.shape == (len(recs), kn.combine_gram_entries(K)) and np.array_equal(a.view(np.int64), b.view(np.int64))
        assert np.all(a[0] == 0)
        for g in range(1, len(recs)):
            _check_gram(a[g], P, Qs, recs[g], K)


@pytest.mark.gpu
def test_gram_kernel_rejects_unsupported_shapes():
    import torch
    from ultrare_b200 import kernels as kn
    dev = _dev()
    rec = torch.zeros((4, 4), dtype=torch.int32, device=dev)
    P = torch.zeros((4, 16), device=dev)
    with pytest.raises(RuntimeError, match="code -2"):
        kn.combine_gram(P, [P] * 65, [rec] * 65)
    P24 = torch.zeros((4, 24), device=dev)
    with pytest.raises(RuntimeError, match="code -2"):
        kn.combine_gram(P24, [P24] * 2, [rec] * 2)


@pytest.mark.gpu
@pytest.mark.parametrize("d", (16, 64))
def test_item_wsum_and_group_score_vs_float64(d):
    """T_g = sum_k w_gk Q_k and b_s + P[u].T_s[i] (users in no group: the last slot) against float64."""
    import torch
    from ultrare_b200 import kernels as kn
    dev = _dev()
    rng = np.random.default_rng(40 + d)
    n_user, n_item, K = 2000, 1500, 5
    P = rng.standard_normal((n_user, d), dtype=np.float32)
    Qs = [rng.standard_normal((n_item, d), dtype=np.float32) for _ in range(K)]
    w = np.concatenate([rng.standard_normal((K, K)), np.full((1, K), 1 / K)]).astype(np.float32)
    b = np.append(rng.standard_normal(K), 0).astype(np.float32)
    Qd = [torch.from_numpy(q).to(dev) for q in Qs]
    T = kn.item_wsum(Qd, torch.from_numpy(w).to(dev))
    T64 = ocomb.item_tables(Qs, w.astype(np.float64))
    tol = 1e-6 * ocomb.item_tables([np.abs(q) for q in Qs], np.abs(w).astype(np.float64)) + 1e-30
    assert np.all(np.abs(T.cpu().numpy() - T64) <= tol)
    owner = rng.integers(0, K, n_user).astype(np.int32)
    owner[::7] = -1
    rec = _records(rng, n_user, n_item, 100_000, dev)
    h = rec.cpu().numpy()
    score, sse = kn.group_score(torch.from_numpy(P).to(dev), T, torch.from_numpy(b).to(dev),
                                torch.from_numpy(owner).to(dev), rec)
    got = score.cpu().numpy().astype(np.float64)
    want = ocomb.scores(P, Qs, w[:K].astype(np.float64), b[:K].astype(np.float64), owner, h[:, 0], h[:, 1])
    slot = np.where(owner[h[:, 0]] >= 0, owner[h[:, 0]], K)
    scale = np.abs(b[slot]) + (np.abs(P[h[:, 0]]).astype(np.float64) *
                               ocomb.item_tables([np.abs(q) for q in Qs], np.abs(w).astype(np.float64))[slot, h[:, 1]]).sum(1)
    assert np.all(np.abs(got - want) <= 1e-5 * scale)
    assert (owner[h[:, 0]] < 0).any()
    r = h[:, 2].view(np.float32).astype(np.float64)
    assert float(sse.item()) == pytest.approx(((got - r) ** 2).sum(), rel=1e-9)


# ------------------------------------------------------------------------------ GPU: Sisa
class _ThreadDist:
    """Ranks of one process as threads on one GPU (as in test_gpu_recommend.py): the collectives Sisa uses, through
    shared slots summed in rank order."""

    def __init__(self, rank, world, shared):
        self.rank, self.world, self.sh = rank, world, shared

    def owner_of_shard(self, s):
        return s % self.world

    def my_shards(self, ids):
        return [s for s in ids if s % self.world == self.rank]

    def _exchange(self, t):
        import torch
        torch.cuda.synchronize()
        self.sh["slots"][self.rank] = t.clone()
        torch.cuda.synchronize()
        self.sh["barrier"].wait()
        parts = list(self.sh["slots"])
        self.sh["barrier"].wait()
        return parts

    def all_reduce(self, t, op="sum"):
        parts = self._exchange(t)
        acc = parts[0].clone()
        for x in parts[1:]:
            acc += x
        t.copy_(acc)
        return t

    def all_gather_into(self, out, part):
        import torch
        out.copy_(torch.cat(self._exchange(part)))
        return out


def _on_ranks(sisa, world, fn):
    """fn(rank view of `sisa`) on `world` threads: rank r keeps the shards s with s % world == r and placeholders for
    the others, as after a multi-GPU pass; returns every rank's result."""
    from ultrare_b200.method.sisa import Sisa, _RemoteModel
    shared = dict(barrier=threading.Barrier(world), slots=[None] * world)
    out, errs = [None] * world, []

    def run(r):
        try:
            sr = Sisa.__new__(Sisa)
            sr.__dict__.update(sisa.__dict__)
            sr.dist = _ThreadDist(r, world, shared)
            P = sisa.model_list[0].user_mat.weight
            sr.model_list = [m if k % world == r else _RemoteModel(P) for k, m in enumerate(sisa.model_list)]
            out[r] = fn(sr)
        except BaseException as e:          # noqa: BLE001 -- re-raised below; the other ranks are released
            errs.append(e)
            shared["barrier"].abort()

    th = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    if errs:
        raise errs[0]
    return out


def _bits(t):
    import torch
    return t.view(torch.int32) if t.dtype == torch.float32 else t


@pytest.mark.gpu
def test_sisa_fit_learn_unlearn_vs_oracle_and_ranks(toy):
    """Toy data, learn -> unlearn with combine='fit' (and 'mean' for the tables):
    * the trained tables are bit-identical to a 'mean' run, and the mean's log0 metrics are unchanged;
    * the unlearn pass's combined test scores equal the oracle fitted on oracle/sisa.read_rating's retained rows
      (<= 1e-4 absolute), and every group's training SSE under the fit is <= that under the mean weights (+ the ridge);
    * recommend equals the per-group oracle top-N (tie rule and near-tie tolerance of test_gpu_recommend.py);
    * as 2 and 3 ranks (threads), the weights, T, lists and scores are bit-equal to one GPU, the metrics equal to
      1e-12 (the ranks add their partial fp64 sums in another order than one GPU's atomics)."""
    import torch
    from test_gpu_recommend import _check, _Param, _sisa_inputs
    from ultrare_b200 import kernels as kn
    from ultrare_b200.method.sisa import Sisa
    dev = _dev()
    z = load_gold("toy_sisa.npz")
    K, n_user = int(z["K"]), toy["n_user"]
    del_user = list(z["del_user"])
    runs = {}
    for combine in ('mean', 'fit'):
        models, passes = [], []
        for is_del in (False, True):
            tl, sl, total, idx, train = _sisa_inputs(toy, z, is_del, K)
            s = Sisa(_Param(2), 'mf', K, idx)
            s.epoch_eval = 'none'
            s.combine = combine
            models = s.unlearn(models, tl, sl, total, del_user, 0, '') if is_del else s.learn(tl, sl, total, 0, '')
            passes.append((s, tl, sl, total, idx, dict(s.final_log),
                           s.model_list[0].user_mat.weight.data.clone(),
                           [m.item_mat.weight.data.clone() for m in s.model_list]))
        runs[combine] = passes
    for p in range(2):
        a, b = runs['mean'][p], runs['fit'][p]
        assert torch.equal(a[6], b[6]) and all(torch.equal(x, y) for x, y in zip(a[7], b[7]))
        assert a[0].combination is None and b[0].combination is not None
    s, tl, sl, total, idx, log, P, Qs = runs['fit'][1]
    P_h, Q_h = P.cpu().numpy(), [q.cpu().numpy() for q in Qs]
    u, i, r = toy["train"]
    kept, gidx = osisa.read_rating(u, i, r, n_user, 5, del_user, K, osisa.uniform_groups(n_user, K), 'a')
    assert [list(g) for g in gidx] == [list(g) for g in idx]
    w_o, b_o = ocomb.fit(P_h, Q_h, [(a[0].astype(np.int64), a[1].astype(np.int64), a[2]) for a in kept])
    owner = s._owner_np
    te = total.dataset.records(dev)
    th = te.cpu().numpy()
    got, _ = kn.group_score(P, s.combination.T, s.combination.b_slot, s._owner, te)
    want = ocomb.scores(P_h, Q_h, w_o, b_o, owner, th[:, 0], th[:, 1])
    assert np.abs(got.cpu().numpy() - want).max() <= 1e-4
    for g, a in enumerate(kept):
        X = ocomb.features(P_h, Q_h, a[0].astype(np.int64), a[1].astype(np.int64))
        sse_fit = ((s.combination.b[g] + X @ s.combination.w[g] - a[2]) ** 2).sum()
        sse_mean = ((X.mean(1) - a[2]) ** 2).sum()
        lam = ocomb.RIDGE * (X ** 2).sum() / K
        assert sse_fit <= sse_mean + lam / K + 1e-9 * sse_mean, (g, sse_fit, sse_mean)
    # the final log is the fit's, the 'mean' run's log is the plain mean's
    assert log['total_rmse'] == pytest.approx(np.sqrt(((got.cpu().numpy() - th[:, 2].view(np.float32)) ** 2).mean()),
                                              rel=1e-6)
    assert runs['mean'][1][5]['total_rmse'] != log['total_rmse']

    items, scores = s.recommend(None, 10, exclude=tl)
    train = np.hstack([a for a in kept])
    rec = torch.from_numpy(np.stack([train[0], train[1], train[2], train[2]], 1).astype(np.int32)).to(dev)
    users = np.arange(n_user)
    slot = np.where(owner >= 0, owner, K)
    seen = kn.seen_lists(rec, n_user, toy["n_item"])
    for g in np.unique(slot).tolist():      # per group: ure_topn on T_g (checked as the mean's lists are), then + b_g
        rows = torch.from_numpy(np.flatnonzero(slot == g)).to(dev)
        ug = torch.from_numpy(users[slot == g].astype(np.int32)).to(dev)
        raw_items, raw = kn.recommend_topn(P, s.combination.T[g], ug, 10, 1.0, seen)
        _check(raw_items, raw, P, s.combination.T[g], ug, 10, 1.0, rec)
        assert torch.equal(items[rows], raw_items)
        assert torch.equal(_bits(scores[rows]), _bits(torch.where(raw_items >= 0, raw + s.combination.b_slot[g], raw)))
    oi, ov = ocomb.topn(P_h, Q_h, s.combination.w, s.combination.b, owner, users, 10,
                        orec.seen_sets(rec.cpu().numpy(), n_user))
    assert (items.cpu().numpy() == oi).mean() > 0.99          # fp32 vs fp64: only near-ties may swap
    np.testing.assert_allclose(scores.cpu().numpy(), ov, atol=1e-4)

    request = np.concatenate([np.random.default_rng(12).permutation(n_user)[:700], np.asarray(del_user)])
    one = s.recommend(request, 10, exclude=tl)
    comb = s.combination

    def rank_pass(sr):
        sr._fit_combination(tl, '')
        sr.test(total, 0, '')
        return sr.combination, dict(sr.final_log), sr.recommend(request, 10, exclude=tl)

    for world in (2, 3):
        for rk, (c, lg, lists) in enumerate(_on_ranks(s, world, rank_pass)):
            assert np.array_equal(c.w, comb.w) and np.array_equal(c.b, comb.b), (world, rk)
            assert torch.equal(_bits(c.T), _bits(comb.T)) and torch.equal(_bits(c.b_slot), _bits(comb.b_slot))
            assert torch.equal(lists[0], one[0]) and torch.equal(_bits(lists[1]), _bits(one[1])), (world, rk)
            for key in ('total_rmse', 'total_ndcg', 'total_hr'):
                assert lg[key] == pytest.approx(log[key], rel=1e-12, abs=1e-15), (world, rk, key)


@pytest.mark.gpu
def test_cli_combine_fit_with_interaction_deletions(cuda_dev, tmp_path, monkeypatch):
    """--deltype inter --combine fit --recommend 10: combine.npy in the learn and the unlearn directories (the unlearn
    one = the final model's weights), and the unlearn pass's Gram equals the float64 Gram over the rows the pair filter
    leaves."""
    import torch
    from test_unlearn_interactions import _deletion_pairs, _read_rating, _toy_env
    from ultrare_b200.main import main
    _, _, save = _toy_env(tmp_path, monkeypatch)
    common = ['--dataset', 'toy', '--synth', '--deltype', 'inter', '--epoch', '2', '--worker', '1', '--verbose', '0']
    main(common + ['--group', '0'])
    ins = main(common + ['--group', '3', '--recommend', '10', '--combine', 'fit'])
    gdir = save + '/2/inter/toy_g3'
    for sub in ('MF_emb-ot_sisa_learn', 'MF_emb-ot_sisa_unlearn'):
        c = np.load(f'{gdir}/{sub}/combine.npy')
        assert c.shape == (3, 4) and c.dtype == np.float64 and np.isfinite(c).all(), sub
        assert os.path.exists(f'{gdir}/{sub}/rec10.npy'), sub
    s = ins.last_sisa
    assert s.combine == 'fit'
    assert np.array_equal(np.load(f'{gdir}/MF_emb-ot_sisa_unlearn/combine.npy'), s.combination.table())
    tr = pd.read_csv(ins.param.train_dir, header=None)
    pairs = _deletion_pairs(tr[0].values, tr[1].values, 2)
    kept, _ = _read_rating(tr[0].values, tr[1].values, tr[2].values, ins.param.n_user, 5, (), 3, s.group_index, 'r',
                           del_rating=pairs)
    P = s.model_list[0].user_mat.weight.data
    Qs = [m.item_mat.weight.data for m in s.model_list]
    for g, a in enumerate(kept):
        rec = np.zeros((a.shape[1], 4), dtype=np.int32)
        rec[:, 0], rec[:, 1] = a[0], a[1]
        rec[:, 2] = a[2].astype(np.float32).view(np.int32)
        _check_gram(s.combination.gram[g], P, Qs, torch.from_numpy(rec).to(cuda_dev), 3)
