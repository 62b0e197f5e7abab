"""The evaluation kernels of csrc/eval.cu against float64 and the stable-rule oracle (oracle/evalm.py).

ure_ensemble_score at every width, model count and user-table sharing pattern, at row counts that run the capped
grids' stride loops several times (thresholds from the device's SM count); ure_rank_metrics at every ranking path's
length boundary, with empty segments, ties, the order indirection, and NaN / +-inf / +-0 scores; ure_eval_jobs with
more jobs than the grid has CTAs to spread, so that every job runs in one CTA."""
import numpy as np
import pytest

from oracle import evalm

D_ALL = (8, 16, 32, 64, 128)
SCORE_RTOL = 1e-5                 # of sum_k sum_t |P_k[u,t] Q_k[i,t]| / denom: fp32 products, shuffle tree, K adds
PATTERNS = ("distinct", "shared", "aaba")
# ranking paths: counting (L <= 64), warp arg-max rounds over the staged segment (65..512), counting from global
# memory (> 512); a warp is 32 lanes and the top lists hold 10
SEG_LENS = (1, 2, 9, 10, 11, 31, 32, 33, 63, 64, 65, 66, 96, 97, 511, 512, 513, 1500)
NAN_LENS = (7, 40, 64, 65, 300, 512, 513, 900)


def _num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _user_tables(pool, K, pattern):
    """K user tables: one per model, one shared by all (the SISA merge), or A, A, B, A, A, B, ... (the kernel keeps
    P[u] in registers while consecutive models share the table and must reload it when the pointer changes)."""
    if pattern == "distinct":
        return [pool[k] for k in range(K)]
    if pattern == "shared":
        return [pool[0]] * K
    return [pool[1] if k % 3 == 2 else pool[0] for k in range(K)]


def _records(rng, n, U, I):
    """n test records, users unsorted, ratings in {0.2, ..., 1.0}; the first row names the last user row and the last
    row the last item row (with n = 1 both are the same row)."""
    u, i = rng.integers(0, U, n), rng.integers(0, I, n)
    u[0], i[-1] = U - 1, I - 1
    return u, i, (rng.integers(1, 6, n) / 5).astype(np.float32)


def _score_ref(Ps, Qs, inter, denom):
    """float64 score, its bound SCORE_RTOL * sum_k sum_t |P_k[u,t] Q_k[i,t]| / denom per row, and the median
    |4-wide chunk| of one model's dot product (one lane's share of it), all from the same fp32 tables on the device."""
    import torch
    u, i = inter[:, 0].long(), inter[:, 1].long()
    s = torch.zeros(inter.shape[0], dtype=torch.float64, device=inter.device)
    a = torch.zeros_like(s)
    chunk = None
    for P, Q in zip(Ps, Qs):
        prod = P.double()[u] * Q.double()[i]
        s += prod.sum(1)
        a += prod.abs().sum(1)
        if chunk is None:
            chunk = float(prod.view(prod.shape[0], -1, 4).sum(2).abs().median())
    return s / denom, SCORE_RTOL * a / denom, chunk


def _sse_ref(s64, bound, inter):
    """float64 SSE of the float64 scores, and the bound on a kernel SSE from scores within `bound` of them: the
    kernel's error e differs from e64 by at most eb = bound + the rounding of the fp32 difference score - r, so
    |e^2 - e64^2| <= eb (2 |e64| + eb)."""
    import torch
    r = inter[:, 2].view(torch.float32).double()
    e64 = s64 - r
    eb = bound + 2.0 ** -24 * (s64.abs() + bound + r.abs())
    return (e64 ** 2).sum(), (eb * (2 * e64.abs() + eb)).sum()


def _check_scores(score, sse, s64, bound, inter, what):
    """Scores within the bound of float64; the SSE equal to the kernel's own scores' squared errors in float64
    (relative 1e-12) and within the propagated bound of the float64 truth's."""
    import torch
    err = (score.double() - s64).abs()
    assert bool((err <= bound).all()), f"{what}: score error {float((err / bound).max()):.3g} x bound"
    own = float(((score - inter[:, 2].view(torch.float32)).double() ** 2).sum())    # score - r in fp32, as the kernel
    got = float(sse.item())
    assert abs(got - own) <= 1e-12 * own, f"{what}: sse {got!r} vs its own scores' {own!r}"
    truth, tol = _sse_ref(s64, bound, inter)
    assert abs(got - float(truth)) <= float(tol), f"{what}: sse {got!r} vs float64 {float(truth)!r}"


def _oracle_sums(u, r, s):
    """(sum NDCG@10, sum HR@10, users) of the stable-rule oracle; users grouped by id, rows in file order."""
    if len(u) == 0:
        return np.zeros(3)
    nd, hr = evalm.rank_metrics(u, r, s, kind="stable")
    users = len(np.unique(u))
    return np.array([nd * users, hr * users, users])


def _check_metrics(got, want, what):
    assert got[2] == want[2], f"{what}: {got[2]} users, oracle {want[2]}"
    assert abs(got[0] - want[0]) <= 1e-12 * max(want[0], 1.0), f"{what}: NDCG sum {got[0]!r}, oracle {want[0]!r}"
    assert abs(got[1] - want[1]) <= 1e-12 * max(want[1], 1.0), f"{what}: HR sum {got[1]!r}, oracle {want[1]!r}"


def _padded(t, fill):
    """t as a view one row into a larger allocation whose row 0 is `fill`: a kernel that read before a segment's
    first row would rank padding (and fail the comparison) instead of reading outside the allocation."""
    import torch
    full = torch.empty((t.shape[0] + 1,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    full[0] = fill
    full[1:] = t
    return full[1:]


# ------------------------------------------------------------------------------ CPU: the rule itself
def test_oracle_ranks_nan_first_and_later_index_first_among_equals():
    """The rule the kernel is held to, on a hand-ranked segment: NaN above +inf, then descending value; among equal
    values (NaN with NaN, -0 with +0, tied ratings) the later index first."""
    nan, inf = np.nan, np.inf
    s = np.array([0.5, nan, -0.0, inf, 0.5, -inf, nan, 0.0, 2.0, nan, 1.0])
    r = np.array([1.0, 0.6, 0.6, 0.4, 1.0, 1.0, 0.2, 1.0, 0.6, 0.8, 0.8])
    top_pred = [9, 6, 1, 3, 8, 10, 4, 0, 7, 2]           # NaN 9, 6, 1 | inf | 2 | 1 | 0.5: 4, 0 | +0 7, -0 2 | (-inf)
    top_rating = [7, 5, 4, 0, 10, 9, 8, 2, 1, 3]         # 1.0: 7, 5, 4, 0 | 0.8: 10, 9 | 0.6: 8, 2, 1 | 0.4 | (0.2)
    assert np.argsort(s, kind="stable")[::-1][:10].tolist() == top_pred
    assert np.argsort(r, kind="stable")[::-1][:10].tolist() == top_rating
    # relevance r[top_pred] = .8 .2 .6 .4 .6 .8 1 1 1 .6; hits (>= 0.8) at p = 0, 5, 6, 7, 8; top_rating[1] = 5 (-inf)
    # is not in top_pred, but p = 1 is no hit anyway
    hr = 5 / 10
    dcg = 0.8 + 0.8 / np.log2(6) + 1 / np.log2(7) + 1 / np.log2(8) + 1 / np.log2(9)
    idcg = 1 + sum(1 / np.log2(p + 1) for p in range(1, 10))
    got_hr, got_ndcg = evalm.user_rank_metrics(r, s)
    assert got_hr == hr
    assert abs(got_ndcg - dcg / idcg) < 1e-15


# ------------------------------------------------------------------------------ GPU: ure_ensemble_score
@pytest.mark.gpu
@pytest.mark.parametrize("d", D_ALL)
def test_ensemble_score_vs_float64(cuda_dev, d):
    """Every K in {1, 2, 5, 8} x user-table pattern x n in {1, GPW - 1, GPW + 1, 1001, > 2.5 grid passes + ragged}
    (GPW = records per warp): scores and SSE against float64; the SSE without scores; partial sums over two halves
    of the models (denom 1) + ure_score_finalize at more than 2.5 of its own grid passes."""
    import torch
    from ultrare_b200 import kernels as kn
    rng = np.random.default_rng(100 + d)
    U, I, G = 3001, 2003, d // 4
    gpw = 32 // G
    fin_rows = _num_sms() * 8 * 256               # one pass of ure_score_finalize's capped grid
    score_rows = _num_sms() * 8 * (256 // G)      # one pass of ure_ensemble_score's capped grid (<= fin_rows)
    n_big = int(2.5 * fin_rows) + 37
    assert n_big > 2.5 * score_rows and n_big % score_rows != 0 and (gpw == 1 or n_big % gpw != 0)
    Ppool = [torch.tensor(rng.standard_normal((U, d), dtype=np.float32), device=cuda_dev) for _ in range(8)]
    Qpool = [torch.tensor(rng.standard_normal((I, d), dtype=np.float32), device=cuda_dev) for _ in range(8)]
    for n in sorted({n for n in (1, gpw - 1, gpw + 1, 1001, n_big) if n >= 1}):
        inter = kn.pack_interactions(*_records(rng, n, U, I), cuda_dev)
        for K in (1, 2, 5, 8):
            for pattern in PATTERNS:
                what = f"d={d} n={n} K={K} {pattern}"
                Ps, Qs = _user_tables(Ppool, K, pattern), Qpool[:K]
                s64, bound, chunk = _score_ref(Ps, Qs, inter, float(K))
                # the bound is far below one lane's share of a dot product: a kernel that drops or doubles a chunk,
                # or reduces over the wrong shuffle width, cannot pass (checked where the medians are stable; the
                # tables and the bound are the same at every n)
                assert n < 1000 or float(bound.median()) < 0.01 * chunk / K, what
                score, sse = kn.ensemble_score(Ps, Qs, inter)
                _check_scores(score, sse, s64, bound, inter, what)
                _, sse_only = kn.ensemble_score(Ps, Qs, inter, want_score=False)
                assert abs(sse_only.item() - sse.item()) <= 1e-12 * sse.item(), what
                if K >= 2:
                    h = K // 2
                    s1, _ = kn.ensemble_score(Ps[:h], Qs[:h], inter, denom=1.0)
                    s2, _ = kn.ensemble_score(Ps[h:], Qs[h:], inter, denom=1.0)
                    fin, sse_fin = kn.score_finalize(s1 + s2, inter, float(K))
                    _check_scores(fin, sse_fin, s64, bound, inter, what + " partial sums + finalize")


# ------------------------------------------------------------------------------ GPU: ure_rank_metrics
@pytest.mark.gpu
def test_rank_metrics_path_boundaries_vs_oracle(cuda_dev):
    """Every ranking path's boundary lengths among enough short segments for the capped grid's segment loop to run
    three times, empty segments (users without test rows) between them, heavily tied dyadic scores and ratings;
    rows in user order (identity) and shuffled (the order indirection of ure_user_segments)."""
    import torch
    from ultrare_b200 import kernels as kn
    rng = np.random.default_rng(7)
    n_short = 3 * _num_sms() * 32
    lens = np.concatenate([SEG_LENS, rng.integers(1, 13, n_short)])
    rng.shuffle(lens)
    uid = np.cumsum(rng.integers(1, 3, len(lens)))           # ids skipped in between: empty segments
    n_user = int(uid[-1]) + 3
    u = np.repeat(uid, lens)
    n = len(u)
    r = (rng.integers(1, 6, n) / 5).astype(np.float32)
    s = (rng.integers(-8, 9, n) / 4).astype(np.float32)
    want = _oracle_sums(u, r, s)
    assert want[2] == len(lens)
    inter = kn.pack_interactions(u, np.zeros(n, dtype=np.int64), r, cuda_dev)
    seg = kn.upload_array(np.concatenate([[0], np.cumsum(np.bincount(u, minlength=n_user))]).astype(np.int64), cuda_dev)
    got = kn.rank_metrics(inter, torch.tensor(s, device=cuda_dev), seg).cpu().numpy()
    _check_metrics(got, want, "user order")
    p = rng.permutation(n)
    inter = kn.pack_interactions(u[p], np.zeros(n, dtype=np.int64), r[p], cuda_dev)
    order, seg = kn.user_segments_device(inter, n_user)
    got = kn.rank_metrics(inter, torch.tensor(s[p], device=cuda_dev), seg, order).cpu().numpy()
    _check_metrics(got, _oracle_sums(u[p], r[p], s[p]), "shuffled rows")


def _nan_segments(rng, L):
    """Score vectors of one segment length: 1, 3, exactly 10 and 12 NaNs (capped at L), all NaN, NaN at the first
    row, +-inf and NaN mixed in, +-0 ties; the others tied dyadic values."""
    def base():
        return (rng.integers(-4, 5, L) / 2).astype(np.float32)

    def at(k):
        return rng.choice(L, min(k, L), replace=False)

    out = [np.full(L, np.nan, dtype=np.float32)]           # first: it lands at row 0 of the table
    for c in (1, 3, 10, 12):
        s = base()
        s[at(c)] = np.nan
        out.append(s)
    s = base()
    s[0] = np.nan
    out.append(s)
    s = base()
    x = at(max(3, L // 4))
    s[x[0::3]], s[x[1::3]], s[x[2::3]] = np.inf, -np.inf, np.nan
    out.append(s)
    s = base()
    x = at(max(2, L // 2))
    s[x] = np.where(rng.random(len(x)) < 0.5, np.float32(-0.0), np.float32(0.0))
    out.append(s)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("L", NAN_LENS)
def test_rank_metrics_nan_and_inf_scores_vs_oracle(cuda_dev, L):
    """NaN ranks above every number and ties with every NaN, -0 ties +0, later index first: segments of length L
    with NaN / +-inf / +-0 scores, between short NaN-free ones, the all-NaN segment at row 0; user order and
    shuffled rows agree with the oracle exactly."""
    import torch
    from ultrare_b200 import kernels as kn
    rng = np.random.default_rng(1000 + L)
    parts = []
    for sv in _nan_segments(rng, L):
        parts += [sv, (rng.integers(-4, 5, rng.integers(1, 20)) / 2).astype(np.float32)]
    s = np.concatenate(parts)
    u = np.repeat(np.arange(len(parts)), [len(x) for x in parts])
    n = len(u)
    r = (rng.integers(1, 6, n) / 5).astype(np.float32)
    for shuffle in (False, True):
        p = rng.permutation(n) if shuffle else np.arange(n)
        pad = torch.tensor([0, 0, int(np.float32(1.0).view(np.int32)), 0], dtype=torch.int32, device=cuda_dev)
        inter = _padded(kn.pack_interactions(u[p], np.zeros(n, dtype=np.int64), r[p], cuda_dev), pad)
        score = _padded(torch.tensor(s[p], device=cuda_dev), float("inf"))
        order, seg = kn.user_segments(u[p])
        assert (order is None) == (not shuffle) and seg[0] == 0
        order = None if order is None else _padded(torch.tensor(order, device=cuda_dev), 0)
        got = kn.rank_metrics(inter, score, torch.tensor(seg, device=cuda_dev), order).cpu().numpy()
        _check_metrics(got, _oracle_sums(u[p], r[p], s[p]), f"L={L} shuffled={shuffle}")


@pytest.mark.gpu
def test_eval_jobs_with_nan_user_rows(cuda_dev):
    """A merged user table with NaN rows (what a diverged sliced unlearn leaves): the job's SSE is NaN, its NDCG and
    HR equal the oracle's on the same scores, for segments on every ranking path; a NaN-free job beside it equals
    the single calls."""
    import torch
    from ultrare_b200 import kernels as kn
    rng = np.random.default_rng(31)
    U, I, d, K = 40, 900, 32, 5
    P = rng.standard_normal((U, d), dtype=np.float32)
    P[rng.choice(np.arange(2, U), 8, replace=False)] = np.nan
    P[[1, 7, 11, U - 1]] = np.nan                           # all-NaN segments on every ranking path (lens below)
    Pt = torch.tensor(P, device=cuda_dev)
    Qs = [torch.tensor(rng.standard_normal((I, d), dtype=np.float32), device=cuda_dev) for _ in range(K)]
    lens = rng.integers(1, 30, U)
    lens[[1, 3, 7, 11, 19]] = [600, 70, 300, 12, 513]
    u = rng.permutation(np.repeat(np.arange(U), lens))
    n = len(u)
    i, r = rng.integers(0, I, n), (rng.integers(1, 6, n) / 5).astype(np.float32)
    inter = kn.pack_interactions(u, i, r, cuda_dev)
    order, seg = kn.user_segments_device(inter, U)
    clean = torch.tensor(np.nan_to_num(P), device=cuda_dev)
    got = kn.eval_jobs([([Pt] * K, Qs, inter, order, seg), ([clean] * K, Qs, inter, order, seg)], d).cpu().numpy()
    score, _ = kn.ensemble_score([Pt] * K, Qs, inter)
    s = score.cpu().numpy()
    assert np.array_equal(np.isnan(s), np.isnan(P[u, 0])) and np.isnan(s).any()
    assert np.isnan(got[0, 0])
    _check_metrics(got[0, 1:], _oracle_sums(u, r, s), "NaN rows")
    score, sse = kn.ensemble_score([clean] * K, Qs, inter)
    want = np.concatenate([sse.cpu().numpy(), kn.rank_metrics(inter, score, seg, order).cpu().numpy()])
    np.testing.assert_allclose(got[1], want, rtol=1e-12, atol=0)


# ------------------------------------------------------------------------------ GPU: ure_eval_jobs
def _job_sets(rng, U, I, dev):
    """Test sets for the jobs: one empty, many tiny, three with thousands of rows and more than 8 users (one with a
    user longer than the staged segment, one shuffled with users that have no rows).  (inter, order, seg, u, r)."""
    import torch
    from ultrare_b200 import kernels as kn
    sets = []

    def add(u, shuffle, device_segments=False):
        if shuffle:
            u = rng.permutation(u)
        i = rng.integers(0, I, len(u))
        i[-1] = I - 1
        r = (rng.integers(1, 6, len(u)) / 5).astype(np.float32)
        inter = kn.pack_interactions(u, i, r, dev)
        if device_segments:
            order, seg = kn.user_segments_device(inter, U)
        else:
            order, seg = kn.user_segments(u)
            order = None if order is None else torch.tensor(order, device=dev)
            seg = torch.tensor(seg, device=dev)
        sets.append((inter, order, seg, u, r))

    add(np.repeat(np.arange(40), rng.integers(50, 150, 40)), False)
    add(np.repeat(np.arange(12), [700, 300, 90, 65, 64, 33, 10, 9, 2, 1, 200, 513]), True)
    add(np.sort(rng.choice(U - 1, 4000) // 2 * 2), True, device_segments=True)        # odd ids: no rows
    big = sets[0]
    sets.append((big[0][:0], None, torch.zeros(1, dtype=torch.int64, device=dev), big[3][:0], big[4][:0]))
    for _ in range(250):
        users = rng.choice(U, rng.integers(1, 6), replace=False)
        add(np.sort(np.repeat(users, rng.integers(1, 9, len(users)))), bool(rng.random() < 0.5))
    return sets


@pytest.mark.gpu
@pytest.mark.parametrize("d", D_ALL)
def test_eval_jobs_one_cta_per_job(cuda_dev, d):
    """At least num_sms * 8 jobs (one CTA per job in both kernels), 1..5 models with the user-table patterns, an empty
    test set (its row stays zero), many tiny sets and a few large ones: every job equals its single calls
    (rtol 1e-12), its SSE is within the float64 bound and its NDCG / HR sums equal the oracle's."""
    import torch
    from ultrare_b200 import kernels as kn
    rng = np.random.default_rng(200 + d)
    U, I = 97, 61
    Ppool = [torch.tensor(rng.standard_normal((U, d), dtype=np.float32), device=cuda_dev) for _ in range(5)]
    Qpool = [torch.tensor(rng.standard_normal((I, d), dtype=np.float32), device=cuda_dev) for _ in range(5)]
    sets = _job_sets(rng, U, I, cuda_dev)
    n_jobs = _num_sms() * 8 + 3
    jobs, want, scores, bounds = [], [], [], []
    for x in range(n_jobs):
        inter, order, seg, _, _ = sets[x % len(sets)]
        K = 1 + x % 5
        Ps = _user_tables([Ppool[k] for k in rng.permutation(5)], K, PATTERNS[(x // 5) % 3])
        Qs = [Qpool[k] for k in rng.permutation(5)[:K]]
        jobs.append((Ps, Qs, inter, order, seg))
        score, sse = kn.ensemble_score(Ps, Qs, inter)
        want.append(torch.cat([sse, kn.rank_metrics(inter, score, seg, order)]))
        scores.append(score)
        if inter.shape[0]:
            s64, bound, _ = _score_ref(Ps, Qs, inter, float(K))
            bounds.append(torch.stack(_sse_ref(s64, bound, inter)))
        else:
            bounds.append(torch.zeros(2, dtype=torch.float64, device=cuda_dev))
    got = kn.eval_jobs(jobs, d).cpu().numpy()
    want = torch.stack(want).cpu().numpy()
    bounds = torch.stack(bounds).cpu().numpy()
    scores = [sc.cpu().numpy() for sc in scores]
    assert got.shape == (n_jobs, 4)
    empty = [x for x in range(n_jobs) if sets[x % len(sets)][0].shape[0] == 0]
    assert empty and not got[empty].any()
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)
    assert np.all(np.abs(got[:, 0] - bounds[:, 0]) <= bounds[:, 1])
    for x in range(n_jobs):
        _, _, _, u, r = sets[x % len(sets)]
        _check_metrics(got[x, 1:], _oracle_sums(u, r, scores[x]), f"d={d} job {x}")
