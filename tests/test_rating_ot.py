"""'rating-ot' grouping: balanced OT clustering of the users' sparse rating rows (reference group.py on readSparseMat).

CPU: the sparse matrix and the records the device path is given, the CLI flag, and that the grouping never needs a
`--group 0` run.  GPU: ure_sparse_cost and ure_sparse_centroid_sums against float64 at every kpad boundary, one outer
iteration against exact EMD, the whole clustering against the oracle loop, and the Group / Instance / CLI surface."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import ROOT, load_gold
from oracle import ot as oot

KS = (2, 5, 8, 9, 16, 17, 32, 33, 64, 65, 128)


def _toy_matrix():
    z = load_gold("toy_data.npz")
    r = (z["train_r2"] / 2.0 / 5.0).astype(np.float32)
    return sp.coo_matrix((r, (z["train_u"].astype(np.int64), z["train_i"].astype(np.int64))),
                         shape=(1508, 2071), dtype=np.float32).tocsr()


def _ml1m_matrix():
    from ultrare_b200 import synth
    (u, i, r), _ = synth.ml_like()
    return sp.coo_matrix(((r / 5.0).astype(np.float32), (u, i)), shape=(synth.ML1M["n_user"], synth.ML1M["n_item"]),
                         dtype=np.float32).tocsr()


def _edge_matrix():
    """1 003 users (not a multiple of a CTA's 8 rows) x 5 000 items: users without ratings, one user with 4 500 ratings
    and one with 1 500 (the whole-CTA long-row path), and stored duplicate (user, item) entries, some of them
    straddling the long rows."""
    rng = np.random.default_rng(7)
    n, m = 1003, 5000
    rows, cols = [], []
    for u in range(n):
        c = {3: 4500, 10: 1500}.get(u, 0 if u in (0, 17, 500, 1002) else int(rng.integers(1, 300)))
        rows.append(np.full(c, u))
        cols.append(np.sort(rng.choice(m, c, replace=False)))
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    vals = rng.integers(1, 6, len(rows)).astype(np.float32) / 5
    dup = np.concatenate([rng.choice(len(rows), 400, replace=False), np.flatnonzero(rows == 3)[:50]])
    rows = np.concatenate([rows, rows[dup]])
    cols = np.concatenate([cols, cols[dup]])
    vals = np.concatenate([vals, rng.integers(1, 6, len(dup)).astype(np.float32) / 5])
    order = np.lexsort((cols, rows))
    rows, cols, vals = rows[order], cols[order], vals[order]
    indptr = np.searchsorted(rows, np.arange(n + 1))
    X = sp.csr_matrix((vals, cols.astype(np.int32), indptr), shape=(n, m))     # stored duplicates are kept
    assert X.nnz == len(rows) and not X.has_canonical_format
    return X


# ------------------------------------------------------------------------------ CPU
def test_read_sparse_mat_sums_duplicates_and_the_records_are_scipys(tmp_path):
    """readSparseMat on a CSV with duplicate (user, item) rows equals SciPy's summed matrix, and the records the device
    path uploads decode to the same matrix."""
    from ultrare_b200.method.utils import sparse_records
    from ultrare_b200.read import readSparseMat
    u = np.array([0, 0, 1, 2, 2, 2, 4, 0])
    i = np.array([3, 1, 2, 0, 0, 5, 4, 3])
    r = np.array([5, 4, 3, 1, 2, 5, 4, 1], dtype=np.float64)
    path = tmp_path / "train.csv"
    path.write_text("".join(f"{a},{b},{c}\n" for a, b, c in zip(u, i, r)))
    X = readSparseMat(str(path), 6, 7, 5)
    dense = np.zeros((6, 7), dtype=np.float32)
    for a, b, c in zip(u, i, r):
        dense[a, b] += np.float32(c / 5)
    assert X.dtype == np.float32 and X.shape == (6, 7)
    assert np.array_equal(X.toarray(), dense)
    ref = sp.coo_matrix(((r / 5).astype(np.float32), (u, i)), shape=(6, 7), dtype=np.float32).tocsr()
    assert np.array_equal(X.indptr, ref.indptr) and np.array_equal(X.indices, ref.indices)
    assert np.array_equal(X.data, ref.data)
    rec = sparse_records(X)
    back = sp.coo_matrix((rec[:, 2].view(np.float32), (rec[:, 0], rec[:, 1])), shape=(6, 7)).toarray()
    assert np.array_equal(back, dense) and (rec[:, 3] == 0).all()
    E = _edge_matrix()                                  # stored duplicates travel to the device as separate records
    rec = sparse_records(E)
    assert len(rec) == E.nnz
    back = sp.coo_matrix((rec[:, 2].view(np.float32), (rec[:, 0], rec[:, 1])), shape=E.shape).toarray()
    assert np.array_equal(back, E.toarray())


def test_grouping_flag_and_its_default():
    from ultrare_b200 import main as m
    assert m.parser.parse_args([]).grouping == 'emb-ot'
    assert m.parser.parse_args(['--grouping', 'rating-ot']).grouping == 'rating-ot'
    with pytest.raises(SystemExit):
        m.parser.parse_args(['--grouping', 'rating-km'])


def test_rating_ot_group_index_reads_the_training_file_and_never_user_mat0(tmp_path, monkeypatch):
    """Instance._group_index('rating-ot', K) hands Group the readSparseMat matrix of the training file and never looks
    for user_mat0.npy."""
    import ultrare_b200.config as cfg
    from ultrare_b200.read import readSparseMat
    seen = {}

    class FakeGroup:
        def __init__(self, rating, dataset, user_mat=None):
            seen["rating"], seen["user_mat"] = rating, user_mat

        def grouping(self, dataset, n_group, var, verbose=True):
            seen["var"] = var
            return [list(range(g, 6, n_group)) for g in range(n_group)]

    path = tmp_path / "train.csv"
    path.write_text("0,1,5\n1,2,4\n1,2,1\n5,0,3\n")
    monkeypatch.setattr(cfg, "Group", FakeGroup)
    ins = cfg.Instance.__new__(cfg.Instance)
    ins.param = type("P", (), dict(n_user=6, n_item=3, dataset="toy", train_dir=str(path), max_rating=5))()
    ins.timing = {}

    def no_user_mat():
        raise AssertionError("rating-ot looked for user_mat0.npy")

    ins._user_mat_path = no_user_mat
    g = ins._group_index("rating-ot", 2)
    assert g == [[0, 2, 4], [1, 3, 5]] and seen["var"] == "rating-ot" and seen["user_mat"] is None
    assert sp.issparse(seen["rating"])
    assert np.array_equal(seen["rating"].toarray(), readSparseMat(str(path), 6, 3, 5).toarray())


# ------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def matrices():
    return {"toy": _toy_matrix(), "ml1m": _ml1m_matrix(), "edge": _edge_matrix()}


def _orders(X, dev):
    from ultrare_b200 import kernels as kn
    from ultrare_b200.method.utils import sparse_records
    return kn.sparse_orders(kn.upload_table(sparse_records(X), dev), X.shape[0], X.shape[1])


def _centroids(X, k, seed):
    """k rows of X (a zero cost and the most cancellation for those users) with a little noise on some of them."""
    rng = np.random.default_rng(seed)
    C = X[rng.choice(X.shape[0], k, replace=False)].toarray().astype(np.float32)
    C[::2] += rng.random((len(C[::2]), C.shape[1]), dtype=np.float32) * 0.01
    return C


def _sparse_cost(csr, C, k, dev):
    import torch
    from ultrare_b200 import kernels as kn
    kp = kn.kpad_for(k)
    Ct = np.zeros((C.shape[1], kp), dtype=np.float32)
    Ct[:, :k] = C.T
    cn = np.square(C.astype(np.float64)).sum(axis=1)
    M, inert = kn.sparse_cost(csr, torch.tensor(Ct, device=dev), torch.tensor(cn, device=dev), k, want_inertia=True)
    return M.cpu().numpy(), float(inert.item())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["toy", "ml1m", "edge"])
def test_sparse_cost_vs_float64(cuda_dev, matrices, name):
    X = matrices[name]
    csr, _ = _orders(X, cuda_dev)
    Xd = X.toarray().astype(np.float64)
    xn = np.square(Xd).sum(axis=1)
    C_all = _centroids(X, max(KS), 1)                  # the centroids of k are the first k rows
    M64_all = oot.cost_matrix(Xd, C_all)
    for k in KS:
        C, M64 = C_all[:k], M64_all[:, :k]
        M, inert = _sparse_cost(csr, C, k, cuda_dev)
        bound = 1e-6 * (xn[:, None] + np.square(C.astype(np.float64)).sum(axis=1)[None, :])
        err = np.abs(M[:, :k] - M64)
        assert (err <= bound).all(), (name, k, float((err - bound).max()))
        assert M.shape == (X.shape[0], max(8, 1 << (k - 1).bit_length())) and np.isposinf(M[:, k:]).all(), (name, k)
        in64 = np.maximum(M64.min(axis=1), 0).sum()
        assert abs(inert - in64) <= 1e-6 * in64, (name, k, inert, in64)
        M2, inert2 = _sparse_cost(csr, C, k, cuda_dev)
        assert np.array_equal(M, M2) and inert == inert2


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["toy", "ml1m", "edge"])
def test_sparse_centroid_sums_vs_float64_and_bit_reproducible(cuda_dev, matrices, name):
    import torch
    from ultrare_b200 import kernels as kn
    X = matrices[name]
    _, csc = _orders(X, cuda_dev)
    Xd = X.toarray().astype(np.float64)
    rng = np.random.default_rng(3)
    for k in KS:
        label = rng.integers(0, k, X.shape[0]).astype(np.int32)
        lab = torch.tensor(label, device=cuda_dev)
        sums, cnt = kn.sparse_centroid_sums(csc, lab, k)
        s = sums.cpu().numpy()
        ref = np.stack([Xd[label == j].sum(axis=0) for j in range(k)]).T           # [n_item, k]
        assert s.shape == (X.shape[1], kn.kpad_for(k)) and (s[:, k:] == 0).all()
        assert (np.abs(s[:, :k] - ref) <= 1e-12 * np.abs(ref)).all(), (name, k)
        assert cnt.cpu().numpy().tolist() == np.bincount(label, minlength=k).tolist()
        sums2, _ = kn.sparse_centroid_sums(csc, lab, k)
        assert torch.equal(sums, sums2)


def _opt_cost(M64, k):
    n = M64.shape[0]
    G = oot.emd_lp(np.ones(n) / n, np.ones(k) / k, M64)
    return float((G * M64).sum() * n)


@pytest.mark.gpu
@pytest.mark.parametrize("name,k", [("toy", 2), ("toy", 4), ("ml1m", 5), ("ml1m", 8)])
def test_one_outer_iteration_is_the_exact_emd_optimum(cuda_dev, matrices, name, k):
    """One outer iteration (Sinkhorn + argmax + balanced rounding) against the exact LP: group sizes exactly n/k and the
    assignment's float64 cost within 1e-6 of the optimum (costs, not labels: an fp32 near-tie cannot fail it)."""
    from ultrare_b200.method.utils import ot_cluster_sparse_device
    X = matrices[name]
    n = X.shape[0]
    assert n % k == 0
    np.random.seed(11)
    c0 = X[np.random.choice(n, size=k, replace=False)].toarray()
    _, lab, _, it = ot_cluster_sparse_device(X, k, max_iters=1, centroid0=c0)
    assert it == 1
    assert np.bincount(lab, minlength=k).tolist() == [n // k] * k
    M64 = oot.cost_matrix(X.toarray(), c0)
    got, opt = float(M64[np.arange(n), lab].sum()), _opt_cost(M64, k)
    assert abs(got - opt) <= 1e-6 * opt, (got, opt)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [4, 5])
def test_sparse_clustering_vs_oracle_loop(cuda_dev, matrices, k):
    """The whole clustering against the oracle's outer loop with the float64 Sinkhorn and the oracle's rounding as the
    plan (as test_ot_cluster_vs_oracle_and_reference does for emb-ot), at the fixed schedule.  Both start from the means
    of random users: from single rating rows the first iteration is full of exact cost ties (every user who shares no
    item with a centroid), on which the oracle's rounding gives up (toy, k = 4: sizes 534 / 218 / 377 / 379), so its loop
    would not be the balanced one; that start is checked against exact EMD by the test above.  The product defaults
    (start from random rows) give balanced sizes and the same labels on a second run with the same seed."""
    from ultrare_b200.method.utils import SINKHORN_SCHEDULE, ot_cluster_sparse_device
    X = matrices["toy"]
    Xd = X.toarray()
    n = X.shape[0]

    def sinkhorn_rounded_plan(a, b, M):
        M = np.asarray(M, dtype=np.float64)
        scale = M.min(axis=1).mean()
        g = oot.sinkhorn_log(M, [(e * scale, i) for e, i in SINKHORN_SCHEDULE])[2]
        lab, _ = oot.balance_labels(M.astype(np.float32), np.argmax(g[None, :] - M, axis=1))
        return np.eye(M.shape[1])[lab]

    rng = np.random.default_rng(k)
    c0 = np.stack([Xd[rng.choice(n, 50, replace=False)].mean(axis=0) for _ in range(k)]).astype(np.float32)
    in_o, lab_o, _, _ = oot.ot_cluster(Xd, k, plan_fn=sinkhorn_rounded_plan, centroid0=c0)
    in_f, lab_f, cen_f, _ = ot_cluster_sparse_device(X, k, centroid0=c0, tol=0.0, warm_start=False)
    assert (lab_f == lab_o).mean() >= 0.99
    assert abs(float(in_f) - float(in_o)) / float(in_o) < 1e-4
    assert cen_f.shape == (k, X.shape[1]) and cen_f.dtype == np.float32
    np.random.seed(5)
    _, lab1, _, _ = ot_cluster_sparse_device(X, k)
    np.random.seed(5)
    _, lab2, _, _ = ot_cluster_sparse_device(X, k)
    assert np.array_equal(lab1, lab2)
    for lab in (lab_f, lab1):
        sizes = np.bincount(lab, minlength=k)
        assert set(sizes.tolist()) <= {n // k, -(-n // k)}, sizes


def test_sparse_path_rejects_what_it_does_not_support():
    from ultrare_b200.method.utils import ot_cluster_sparse_device
    with pytest.raises(TypeError):
        ot_cluster_sparse_device(np.zeros((4, 3), dtype=np.float32), 2)
    with pytest.raises(ValueError):
        ot_cluster_sparse_device(sp.csr_matrix((300, 4), dtype=np.float32), 129)


def _point_at_tmp(monkeypatch, tmp_path):
    import ultrare_b200.config as cfg
    import ultrare_b200.group as grp
    data, save = str(tmp_path / "data"), str(tmp_path / "result")
    for mod in (cfg, grp):
        monkeypatch.setattr(mod, "DATA_DIR", data)
        monkeypatch.setattr(mod, "SAVE_DIR", save)
    return data, save


@pytest.mark.gpu
def test_group_grouping_rating_ot_writes_and_reads_its_cache(cuda_dev, tmp_path, monkeypatch):
    import ultrare_b200.config as cfg
    import ultrare_b200.group as grp
    from ultrare_b200 import synth
    from ultrare_b200.read import readSparseMat
    data, _ = _point_at_tmp(monkeypatch, tmp_path)
    synth.ensure_dataset("toy")
    p = cfg.InsParam("toy", 1, 1, [32], 3, 2, "rand")
    X = readSparseMat(p.train_dir, p.n_user, p.n_item, p.max_rating)
    res = grp.Group(X, "toy").grouping("toy", 3, "rating-ot", verbose=False)
    assert len(res) == 3 and all(g == sorted(g) for g in res)
    assert sorted(u for g in res for u in g) == list(range(p.n_user))
    assert {len(g) for g in res} <= {p.n_user // 3, -(-p.n_user // 3)}
    assert os.path.exists(data + "/toy/val/rating-ot3.npy")

    def no_clustering(*a, **kw):
        raise AssertionError("the cached grouping was not read back")

    monkeypatch.setattr(grp, "ot_cluster", no_clustering)
    assert grp.Group(X, "toy").grouping("toy", 3, "rating-ot", verbose=False) == res


@pytest.mark.gpu
def test_instance_run_group_rating_ot_without_a_full_run(cuda_dev, tmp_path, monkeypatch):
    import ultrare_b200.config as cfg
    from ultrare_b200 import synth
    data, save = _point_at_tmp(monkeypatch, tmp_path)
    synth.ensure_dataset("toy")
    p = cfg.InsParam("toy", 2, 1, [32], 3, 2, "rand")
    ins = cfg.Instance(p)
    ins.runGroup(is_save=True, learn_type='sisa', group_type='rating-ot', n_group=3, verbose=0)
    gdir = save + "/2/rand/toy_g3"
    for sub in ("MF_rating-ot_sisa_learn", "MF_rating-ot_sisa_unlearn"):
        l0 = np.load(f"{gdir}/{sub}/log0.npy", allow_pickle=True).item()
        assert np.isfinite(l0['total_rmse']), sub
    cache = np.load(data + "/toy/val/rating-ot3.npy", allow_pickle=True)
    assert sorted(u for g in cache for u in g) == list(range(p.n_user))
    assert not os.path.exists(save + "/2/rand/toy_g0")


@pytest.mark.gpu
def test_cli_rating_ot_end_to_end(cuda_dev, tmp_path):
    env = dict(os.environ, ULTRARE_ROOT=str(tmp_path))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "main.py"), "--dataset", "toy", "--synth", "--group", "3",
                        "--grouping", "rating-ot", "--epoch", "2", "--verbose", "0"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    gdir = tmp_path / "result" / "2" / "rand" / "toy_g3"
    for sub in ("MF_rating-ot_sisa_learn", "MF_rating-ot_sisa_unlearn"):
        assert (gdir / sub / "log0.npy").exists(), sub
    assert (tmp_path / "data" / "toy" / "val" / "rating-ot3.npy").exists()
