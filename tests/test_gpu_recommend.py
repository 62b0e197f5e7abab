"""Top-N recommendation over the whole catalogue: the float64 oracle (oracle/recommend.py) against brute force and a
hand-computed answer (CPU), and the tcgen05 top-N kernel, the seen lists, the metrics kernel and the Python surface
(utils.recommend, Sisa.recommend) against the oracle on the GPU."""
import numpy as np
import pytest

from conftest import init_weights, load_gold
from oracle import recommend as orec

D_ALL = (8, 16, 32, 64, 128)


# ------------------------------------------------------------------------------ CPU: the oracle itself
def test_oracle_topn_matches_brute_force_with_ties():
    """oracle.topn == a plain sort by (-score, item) with seen items removed; integer tables plant many ties."""
    rng = np.random.default_rng(0)
    n_user, n_item, d = 40, 57, 8
    P = rng.integers(-2, 3, (n_user, d)).astype(np.float64)
    S = rng.integers(-2, 3, (n_item, d)).astype(np.float64)
    S[10] = S[3]                                        # identical items: equal scores for every user
    recs = np.stack([rng.integers(0, n_user, 300), rng.integers(0, n_item, 300)], 1)
    seen = orec.seen_sets(recs, n_user)
    users = np.array([5, 0, 5, 39, 17, 3])
    for N in (1, 7, 64):
        items, vals, n_ok = orec.topn(P, S, users, N, 0.5, seen)
        for r, u in enumerate(users):
            cand = [i for i in range(n_item) if i not in seen[u]]
            sc = {i: 0.5 * float(P[u] @ S[i]) for i in cand}
            want = sorted(cand, key=lambda i: (-sc[i], i))[:N]
            got = [int(x) for x in items[r] if x >= 0]
            assert got == want and n_ok[r] == len(cand)
            assert np.all(items[r, len(want):] == -1) and np.all(np.isneginf(vals[r, len(want):]))
            np.testing.assert_array_equal(vals[r, :len(want)], [sc[i] for i in want])


def test_oracle_metrics_known_answer():
    """Hand-computed HR / Recall / NDCG: a user without relevant items (skipped), |rel| > N, a hit at position 0,
    a duplicated relevant test item counted once."""
    N = 3
    items = np.array([[7, 1, 2],       # user 0: rel {7, 2}: hits at 0 and 2
                      [4, 5, 6],       # user 1: no relevant item -> not counted
                      [9, 8, -1],      # user 2: rel {1, 2, 3, 8} (|rel| > N): hit at 1
                      [0, 1, 2]])      # user 3: rel {5}: no hit
    test = np.array([[0, 7, 1.0], [0, 2, 0.8], [0, 3, 0.6], [1, 4, 0.6], [2, 1, 1.0], [2, 2, 0.8], [2, 3, 1.0],
                     [2, 8, 0.8], [2, 8, 1.0], [3, 5, 0.8]])
    m = orec.metrics(items, np.arange(4), test, N)
    w = 1 / np.log2(np.arange(2, 5))
    assert m["users"] == 3
    assert m["hr"] == pytest.approx(2.0)
    assert m["recall"] == pytest.approx(2 / 2 + 1 / 4 + 0)
    assert m["ndcg"] == pytest.approx((w[0] + w[2]) / (w[0] + w[1]) + w[1] / w.sum() + 0)


# ------------------------------------------------------------------------------ GPU helpers
def _dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _seen_mask(recs, users, n_item):
    """bool [m, n_item] on the device: item i seen by the user of request row r."""
    import torch
    m = users.shape[0]
    mask = torch.zeros((m, n_item), dtype=torch.bool, device=users.device)
    if recs is None or recs.shape[0] == 0:
        return mask
    ru, ri = recs[:, 0].long(), recs[:, 1].long()
    order = torch.argsort(ru, stable=True)
    ru, ri = ru[order], ri[order]
    start = torch.searchsorted(ru, users.long())
    stop = torch.searchsorted(ru, users.long(), right=True)
    cnt = stop - start
    rows = torch.repeat_interleave(torch.arange(m, device=users.device), cnt)
    offs = torch.arange(int(cnt.sum()), device=users.device) - torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
    mask[rows, ri[torch.repeat_interleave(start, cnt) + offs]] = True
    return mask


def _check(items, scores, P, S, users, N, scale, recs=None):
    """The kernel's lists against the float64 scores: scores within 1e-5 * sum_t |P S| * scale, seen items absent,
    distinct items, sorted under the tie rule, padding exactly where fewer than N items are eligible, and every eligible
    item left out scored no higher than the lowest returned one (plus the tolerance)."""
    import torch
    U = users.long()
    P64, S64 = P.double()[U], S.double()
    s64 = (P64 @ S64.T) * scale
    tol = 1e-5 * (P64.abs() @ S64.abs().T) * scale + 1e-30
    elig = ~_seen_mask(recs, users, S.shape[0])
    n_elig = elig.sum(1)
    valid = items >= 0
    n_valid = valid.sum(1)
    assert torch.equal(n_valid, torch.clamp(n_elig, max=N)), "wrong list length"
    assert torch.equal(valid, torch.arange(N, device=items.device)[None, :] < n_valid[:, None]), "padding not at the end"
    assert torch.isneginf(scores[~valid]).all()
    idx = items.clamp(min=0).long()
    g, t = s64.gather(1, idx), tol.gather(1, idx)
    assert ((scores.double() - g).abs() <= t)[valid].all(), "score outside tolerance"
    assert elig.gather(1, idx)[valid].all(), "seen item returned"
    si = torch.sort(torch.where(valid, items, -1 - torch.arange(N, device=items.device)[None, :]), 1).values
    assert (si[:, 1:] != si[:, :-1]).all(), "item returned twice"
    a, b = scores[:, :-1], scores[:, 1:]
    ok = (a > b) | ((a == b) & (items[:, :-1] < items[:, 1:]))
    assert (ok | ~valid[:, 1:]).all(), "list not sorted under the tie rule"
    left = elig.clone()
    left.scatter_(1, idx, False)
    lo = torch.where(valid, g, torch.full_like(g, float("inf"))).min(1).values
    lo_tol = torch.where(valid, t, torch.zeros_like(t)).max(1).values
    worst = torch.where(left, s64 - tol, torch.full_like(s64, -float("inf"))).max(1).values
    full = n_valid == N
    assert (worst[full] <= (lo + lo_tol)[full]).all(), "an eligible item better than the list was left out"


def _tables(rng, n_user, n_item, d, dev):
    import torch
    P = torch.from_numpy(rng.standard_normal((n_user, d), dtype=np.float32)).to(dev)
    S = torch.from_numpy(rng.standard_normal((n_item, d), dtype=np.float32)).to(dev)
    return P, S


def _random_records(rng, n_user, n_item, n, dev):
    import torch
    r = np.zeros((n, 4), dtype=np.int32)
    r[:, 0] = rng.integers(0, n_user, n)
    r[:, 1] = rng.integers(0, n_item, n)
    r[:, 2] = np.float32(0.8).view(np.int32)
    return torch.from_numpy(r).to(dev)


# ------------------------------------------------------------------------------ GPU: kernels
@pytest.mark.gpu
def test_seen_lists_are_sorted_csr_of_the_records():
    import torch
    from ultrare_b200 import kernels as kn
    dev = _dev()
    rng = np.random.default_rng(1)
    for n_user, n_item, n in ((300, 70000, 20000), (1, 5, 3), (70000, 300, 50000)):
        recs = _random_records(rng, n_user, n_item, n, dev)
        off, items = kn.seen_lists([recs[: n // 2], recs[n // 2:]], n_user, n_item)
        h = recs.cpu().numpy()
        order = np.lexsort((h[:, 1], h[:, 0]))
        np.testing.assert_array_equal(items.cpu().numpy(), h[order, 1])
        np.testing.assert_array_equal(off.cpu().numpy(), np.concatenate([[0], np.cumsum(np.bincount(h[:, 0], minlength=n_user))]))


@pytest.mark.gpu
@pytest.mark.parametrize("d", D_ALL)
def test_topn_kernel_vs_oracle(d):
    """Every d: m not a multiple of 128 (1 and 300 rows, permuted, with duplicates), n_item in {1, 2071, 3416},
    N in {1, 10, 64} (N > eligible items pads), seen items excluded."""
    import torch
    from ultrare_b200 import kernels as kn
    dev = _dev()
    rng = np.random.default_rng(d)
    n_user = 500
    for n_item in (1, 2071, 3416):
        P, S = _tables(rng, n_user, n_item, d, dev)
        recs = _random_records(rng, n_user, n_item, 20 * n_user, dev)
        seen = kn.seen_lists(recs, n_user, n_item)
        u300 = rng.permutation(n_user)[:300]
        u300[::7] = u300[3]                              # duplicates
        for users in (np.array([int(rng.integers(n_user))]), u300):
            ut = torch.from_numpy(users.astype(np.int32)).to(dev)
            for N in (1, 10, 64):
                for sn, r in ((None, None), (seen, recs)):
                    items, scores = kn.recommend_topn(P, S, ut, N, 0.25, sn)
                    _check(items, scores, P, S, ut, N, 0.25, r)


@pytest.mark.gpu
@pytest.mark.parametrize("d", (16, 64, 128))
def test_topn_exact_tie_rule_on_dyadic_inputs(d):
    """Small integers: every product and sum is exact in fp32, so the lists equal the oracle's exactly, including
    the planted ties (identical item rows) that only the item id orders."""
    import torch
    from ultrare_b200 import kernels as kn
    dev = _dev()
    rng = np.random.default_rng(10 + d)
    n_user, n_item = 700, 3000
    P = rng.integers(-3, 4, (n_user, d)).astype(np.float32)
    S = rng.integers(-3, 4, (n_item, d)).astype(np.float32)
    S[rng.integers(0, n_item, 1500)] = S[rng.integers(0, 40, 1500)]     # many identical rows
    P[:, d // 2:] = 0                                                     # fewer distinct scores, more ties
    recs = _random_records(rng, n_user, n_item, 30000, dev)
    users = rng.permutation(n_user)[:333].astype(np.int32)
    seen_sets = orec.seen_sets(recs.cpu().numpy(), n_user)
    for N in (1, 10, 64):
        items, scores = kn.recommend_topn(torch.from_numpy(P).to(dev), torch.from_numpy(S).to(dev),
                                          torch.from_numpy(users).to(dev), N, 0.25, kn.seen_lists(recs, n_user, n_item))
        oi, ov, _ = orec.topn(P, S, users, N, 0.25, seen_sets)
        np.testing.assert_array_equal(items.cpu().numpy(), oi)
        np.testing.assert_array_equal(scores.cpu().numpy().astype(np.float64), ov)


@pytest.mark.gpu
def test_topn_exclusion_on_the_toy_training_set(toy):
    """Exclusion = the toy training records; a user who has seen every item gets an all -1 list."""
    import torch
    from ultrare_b200 import kernels as kn
    from ultrare_b200.method.utils import recommend, MF
    dev = _dev()
    n_user, n_item = toy["n_user"], toy["n_item"]
    u, i, r = toy["train"]
    rec = np.zeros((len(u) + n_item, 4), dtype=np.int32)
    rec[:len(u), 0], rec[:len(u), 1] = u, i
    rec[len(u):, 0], rec[len(u):, 1] = 7, np.arange(n_item)            # user 7 has seen everything
    recs = torch.from_numpy(rec).to(dev)
    P0, Q0 = init_weights(5)
    model = MF.from_weights(P0, Q0)
    items, scores = recommend([model], None, 10, exclude=recs)
    assert (items[7] == -1).all() and torch.isneginf(scores[7]).all()
    users = torch.arange(n_user, dtype=torch.int32, device=dev)
    _check(items, scores, model.user_mat.weight, model.item_mat.weight, users, 10, 1.0, recs)
    oi, ov, _ = orec.topn(P0, Q0, np.arange(0, n_user, 37), 10, 1.0, orec.seen_sets(rec, n_user))
    got = items.cpu().numpy()[::37]
    assert (got == oi).mean() > 0.99          # fp32 vs fp64: only near-ties may swap


@pytest.mark.gpu
def test_topn_c3_shaped_catalogue_sampled_against_float64():
    """138 493 users x 26 744 items, d = 64: every user recommended, 512 sampled rows checked against a float64
    product on the GPU."""
    import torch
    from ultrare_b200 import kernels as kn
    dev = _dev()
    rng = np.random.default_rng(3)
    n_user, n_item, d = 138493, 26744, 64
    P, S = _tables(rng, n_user, n_item, d, dev)
    recs = _random_records(rng, n_user, n_item, 2_000_000, dev)
    users = torch.arange(n_user, dtype=torch.int32, device=dev)
    items, scores = kn.recommend_topn(P, S, users, 10, 0.2, kn.seen_lists(recs, n_user, n_item))
    pick = torch.from_numpy(rng.choice(n_user, 512, replace=False)).to(dev)
    _check(items[pick], scores[pick], P, S, users[pick], 10, 0.2, recs)


@pytest.mark.gpu
def test_topn_single_user_over_a_million_items_is_split_and_deterministic():
    """m = 1, 10^6 items, d = 128: the item range is split over CTAs and merged; two calls are bit-identical."""
    import torch
    from ultrare_b200 import _lib, kernels as kn
    dev = _dev()
    rng = np.random.default_rng(4)
    n_item, d = 1_000_000, 128
    P, S = _tables(rng, 3, n_item, d, dev)
    users = torch.tensor([1], dtype=torch.int32, device=dev)
    assert _lib.lib().ure_topn_scratch_bytes(1, n_item, d, 64) > 0          # the split path
    recs = _random_records(rng, 3, n_item, 50000, dev)
    seen = kn.seen_lists(recs, 3, n_item)
    a = kn.recommend_topn(P, S, users, 64, 1.0, seen)
    b = kn.recommend_topn(P, S, users, 64, 1.0, seen)
    _check(a[0], a[1], P, S, users, 64, 1.0, recs)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int32), b[1].view(torch.int32))
    u2 = torch.from_numpy(rng.integers(0, 3, 1000).astype(np.int32)).to(dev)
    c = kn.recommend_topn(P, S[:300000], u2, 10, 1.0)
    e = kn.recommend_topn(P, S[:300000], u2, 10, 1.0)
    assert torch.equal(c[0], e[0]) and torch.equal(c[1].view(torch.int32), e[1].view(torch.int32))


@pytest.mark.gpu
def test_topn_rejects_unsupported_shapes():
    import torch
    from ultrare_b200 import kernels as kn
    dev = _dev()
    P = torch.zeros((4, 16), device=dev)
    u = torch.zeros(2, dtype=torch.int32, device=dev)
    for N in (0, 65):
        with pytest.raises(RuntimeError, match="code -2"):
            kn.recommend_topn(P, P, u, N, 1.0)
    with pytest.raises(RuntimeError, match="code -2"):
        kn.recommend_topn(torch.zeros((4, 24), device=dev), torch.zeros((4, 24), device=dev), u, 5, 1.0)


@pytest.mark.gpu
def test_topn_metrics_kernel_vs_oracle():
    import torch
    from ultrare_b200 import kernels as kn
    from ultrare_b200.method.utils import topn_metrics
    dev = _dev()
    rng = np.random.default_rng(6)
    n_user, n_item, N = 900, 200, 20
    m = 1200
    users = rng.integers(0, n_user, m).astype(np.int32)
    items = np.stack([rng.permutation(n_item)[:N] for _ in range(m)]).astype(np.int32)
    items[::5, N - 4:] = -1
    n = 30000
    test = np.zeros((n, 4), dtype=np.int32)
    test[:, 0] = rng.integers(0, n_user, n)
    test[:, 1] = rng.integers(0, n_item, n)
    test[:, 2] = (rng.integers(1, 6, n).astype(np.float32) / 5).view(np.int32)
    t = torch.from_numpy(test).to(dev)
    out = kn.topn_metrics(torch.from_numpy(items).to(dev), torch.from_numpy(users).to(dev), t, n_user).cpu().numpy()
    host = np.stack([test[:, 0], test[:, 1], test[:, 2].view(np.float32)], 1).astype(np.float64)
    for N_ in (N, 7):
        want = orec.metrics(items, users, host, N_)
        got = kn.topn_metrics(torch.from_numpy(np.ascontiguousarray(items[:, :N_])).to(dev),
                              torch.from_numpy(users).to(dev), t, n_user).cpu().numpy()
        np.testing.assert_allclose(got, [want["hr"], want["recall"], want["ndcg"], want["users"]], rtol=1e-12)
    met = topn_metrics(torch.from_numpy(items).to(dev), users, t, N)
    assert met["users"] == int(out[3]) and met["hr"] == pytest.approx(out[0] / out[3])


def _sisa_inputs(toy, z, is_del, K):
    from ultrare_b200.read import RatingData, loadData, readRating
    import pandas as pd
    from oracle import sisa as osisa
    n_user = toy["n_user"]
    tr = pd.DataFrame({0: toy["train"][0], 1: toy["train"][1], 2: toy["train"][2]})
    te = pd.DataFrame({0: toy["test"][0], 1: toy["test"][1], 2: toy["test"][2]})
    trr, idx = readRating(tr, n_user, 5, list(z["del_user"]) if is_del else [], [], K, osisa.uniform_groups(n_user, K), 'a')
    ter, _ = readRating(te, n_user, 5, [], [], K, idx)
    tl = [loadData(RatingData(trr[s]), 3000, 1, True) for s in range(K)]
    sl = [loadData(RatingData(ter[s]), 3000, 1, False) for s in range(K)]
    total = loadData(RatingData(np.hstack(ter)), 3000, 1, False)
    return tl, sl, total, idx, np.hstack(trr)


class _Param:
    def __init__(self, epochs, n_user=1508, n_item=2071):
        self.n_user, self.n_item, self.k, self.lam = n_user, n_item, 16, 0.1
        self.seed, self.lr, self.lr_decay, self.momentum = 42, 0.001, 0.95, 0.9
        self.epochs, self.batch = epochs, 3000


class _ThreadDist:
    """Ranks of one process as threads on one GPU: the collectives Sisa.recommend uses, through shared slots (sums in
    rank order) -- the multi-GPU branch runs without a second GPU."""

    def __init__(self, rank, world, shared):
        self.rank, self.world, self.sh = rank, world, shared

    def owner_of_shard(self, s):
        return s % self.world

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


def _recommend_on_ranks(sisa, world, users, top_n, exclude):
    """Sisa.recommend of `sisa`'s model_list as `world` ranks (threads): rank r keeps the shards s with s % world == r
    and placeholders for the others, as after a multi-GPU learn; returns every rank's (items, scores)."""
    import threading
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
            out[r] = sr.recommend(users, top_n, exclude=exclude)
        except BaseException as e:          # noqa: BLE001 -- re-raised below; the other rank is released
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


def _bit_equal(a, b):
    import torch
    return torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int32), b[1].view(torch.int32))


@pytest.mark.gpu
def test_sisa_learn_unlearn_recommend_and_scratch_vs_oracle(toy):
    """Sisa.learn then Sisa.unlearn on the toy data; after each, Sisa.recommend (seen = that pass's training data)
    equals the oracle on model_list's tables and, bit for bit, utils.recommend on the same tables and the multi-rank
    branch run as two and three ranks (threads on one GPU; a permuted request with duplicates, deleted users -- in no
    group after the unlearn -- included).  After the unlearn, deleted users' lists hold items they had seen before the
    deletion.  utils.recommend of a Scratch model too."""
    import torch
    from ultrare_b200.method.scratch import Scratch
    from ultrare_b200.method.sisa import Sisa
    from ultrare_b200.method.utils import recommend
    from ultrare_b200.read import RatingData, loadData
    dev = _dev()
    z = load_gold("toy_sisa.npz")
    K = int(z["K"])
    n_user = toy["n_user"]
    users = torch.arange(n_user, dtype=torch.int32, device=dev)
    rng = np.random.default_rng(12)
    request = rng.permutation(n_user)[:700]
    request[::9] = request[5]
    request = np.concatenate([request, np.asarray(z["del_user"])])
    deleted = np.asarray(z["del_user"], dtype=np.int64)
    models, learn_train, tl_learn = [], None, None
    for is_del in (False, True):
        tl, sl, total, idx, train = _sisa_inputs(toy, z, is_del, K)
        s = Sisa(_Param(2), 'mf', K, idx)
        s.epoch_eval = 'none'
        models = s.unlearn(models, tl, sl, total, list(z["del_user"]), 0, '') if is_del else s.learn(tl, sl, total, 0, '')
        items, scores = s.recommend(None, 10, exclude=tl)
        P = s.model_list[0].user_mat.weight.data
        Ssum = sum(m.item_mat.weight.data.double() for m in s.model_list).float()
        rec = torch.from_numpy(np.stack([train[0], train[1], train[2], train[2]], 1).astype(np.int32)).to(dev)
        _check(items, scores, P, Ssum, users, 10, 1.0 / K, rec)
        assert _bit_equal((items, scores), recommend(s.model_list, None, 10, exclude=tl))
        one = s.recommend(request, 10, exclude=tl)
        for world in (2, 3):
            for r, got in enumerate(_recommend_on_ranks(s, world, request, 10, tl)):
                assert _bit_equal(got, one), f"world {world}, rank {r} differs from one GPU"
        if not is_del:
            learn_train, tl_learn = train, tl
            continue
        # the deleted users are gone from this pass's training data, so the items they had seen before are eligible
        assert not set(deleted.tolist()) & set(train[0].astype(int).tolist())
        old = {int(u): set(learn_train[1][learn_train[0] == u].astype(int).tolist()) for u in deleted}
        d_items, d_scores = s.recommend(deleted, 64, exclude=tl)
        _check(d_items, d_scores, P, Ssum, torch.from_numpy(deleted.astype(np.int32)).to(dev), 64, 1.0 / K, rec)
        got = d_items.cpu().numpy()
        assert sum(len(set(got[r].tolist()) & old[int(u)]) for r, u in enumerate(deleted)) > 0
        before = s.recommend(deleted, 64, exclude=tl_learn)[0].cpu().numpy()      # their old items excluded again
        assert sum(len(set(before[r].tolist()) & old[int(u)]) for r, u in enumerate(deleted)) == 0
    sc = Scratch(_Param(2), 'mf')
    tr = loadData(RatingData(np.stack([toy["train"][0], toy["train"][1], toy["train"][2] / 5.0]).astype(np.float64)),
                  3000, 1, True)
    te = loadData(RatingData(np.stack([toy["test"][0], toy["test"][1], toy["test"][2] / 5.0]).astype(np.float64)),
                  3000, 1, False)
    model = sc.train(tr, te, [], 0, '')
    items, scores = recommend([model], None, 10, exclude=tr)
    rec = tr.dataset.records(dev)
    _check(items, scores, model.user_mat.weight.data, model.item_mat.weight.data, users, 10, 1.0, rec)
    with pytest.raises(ValueError):
        other = type(model).from_weights(*init_weights(9))
        recommend([model, other], [0, 1], 10)


@pytest.mark.gpu
def test_out_of_range_inputs_are_rejected():
    """Seen-list records with ids outside the tables raise (the radix passes are sized by them); metrics of lists
    wider than 64 are URE_EUNSUPPORTED (the position weights stop there)."""
    import torch
    from ultrare_b200 import kernels as kn
    dev = _dev()
    rng = np.random.default_rng(13)
    for bad in ((0, 50), (0, -1), (10, 0), (-1, 0)):
        recs = _random_records(rng, 10, 50, 100, dev)
        recs[7, 0], recs[7, 1] = bad
        with pytest.raises(ValueError):
            kn.seen_lists(recs, 10, 50)
    test = _random_records(rng, 10, 50, 100, dev)
    u = torch.arange(10, dtype=torch.int32, device=dev)
    assert kn.topn_metrics(torch.zeros((10, 64), dtype=torch.int32, device=dev), u, test, 10)[3] >= 0
    with pytest.raises(RuntimeError, match="code -2"):
        kn.topn_metrics(torch.zeros((10, 65), dtype=torch.int32, device=dev), u, test, 10)


# ------------------------------------------------------------------------------ GPU: two ranks over NCCL
def _toy_dict():
    zt = load_gold("toy_data.npz")
    out = {p: (zt[p + "_u"].astype(np.int64), zt[p + "_i"].astype(np.int64), zt[p + "_r2"].astype(np.float64) / 2.0)
           for p in ("train", "test")}
    out["n_user"], out["n_item"] = 1508, 2071
    return out


def _nccl_learn_unlearn_recommend(dist_obj, request):
    """learn -> recommend, unlearn -> recommend on toy as one rank of `dist_obj`; the merged user table, this rank's
    item tables and the lists of every pass."""
    import torch
    from ultrare_b200.method.sisa import Sisa
    toy, z = _toy_dict(), load_gold("toy_sisa.npz")
    K = int(z["K"])
    out, models = [], []
    for is_del in (False, True):
        tl, sl, total, idx, _ = _sisa_inputs(toy, z, is_del, K)
        s = Sisa(_Param(2), 'mf', K, idx)
        s.init_on_device = False
        s.epoch_eval = 'none'
        s.dist = dist_obj
        models = s.unlearn(models, tl, sl, total, list(z["del_user"]), 0, '') if is_del else s.learn(tl, sl, total, 0, '')
        items, scores = s.recommend(request, 10, exclude=tl)
        out.append(dict(P=s.model_list[0].user_mat.weight.data.cpu().numpy(), items=items.cpu().numpy(),
                        scores=scores.cpu().numpy(),
                        Q={k: m.item_mat.weight.data.cpu().numpy() for k, m in enumerate(s.model_list)
                           if getattr(m, 'item_mat', None) is not None}))
    torch.cuda.synchronize()
    return out


def _nccl_worker(rank, world, port, request, q):
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from ultrare_b200 import dist as udist
    d = udist.init_from_env(backend="nccl")
    res = _nccl_learn_unlearn_recommend(d, request)
    d.barrier()
    q.put((rank, res))
    d.td.destroy_process_group()


@pytest.mark.gpu
def test_two_rank_sisa_recommend_equals_one_gpu_on_the_same_tables():
    """Two ranks over NCCL (skipped with fewer than 2 GPUs): learn -> recommend and unlearn -> recommend; both ranks
    return the same lists, equal bit for bit to utils.recommend on one GPU over the same tables (gathered from the
    ranks) with the same seen items."""
    import socket
    import torch
    import torch.multiprocessing as mp
    from conftest import collect_results
    from ultrare_b200.method.utils import MF, recommend
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    dev = torch.device("cuda:0")
    z = load_gold("toy_sisa.npz")
    K = int(z["K"])
    request = np.concatenate([np.random.default_rng(14).permutation(1508)[:600], np.asarray(z["del_user"])])
    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, request, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = collect_results(procs, q, 2, timeout=300)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    toy = _toy_dict()
    for phase, is_del in ((0, False), (1, True)):
        tl = _sisa_inputs(toy, z, is_del, K)[0]
        Q = {**res[0][phase]["Q"], **res[1][phase]["Q"]}
        assert sorted(Q) == list(range(K))
        P = res[0][phase]["P"]
        assert np.array_equal(P, res[1][phase]["P"])
        models = [MF.from_weights(P, Q[k], device=dev) for k in range(K)]
        items, scores = recommend(models, request, 10, exclude=tl)
        for r in range(2):
            assert np.array_equal(res[r][phase]["items"], items.cpu().numpy())
            assert np.array_equal(res[r][phase]["scores"].view(np.int32), scores.cpu().numpy().view(np.int32))
