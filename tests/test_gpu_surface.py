"""GPU parity of the drop-in Python surface (Scratch / Sisa / Group / Instance) against the
fixtures the reference itself produced on its toy data (tests/golden/, oracle/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from conftest import init_weights, load_gold
from oracle import mf as omf, ot as oot, sisa as osisa

pytestmark = pytest.mark.gpu
N_USER, N_ITEM, BATCH, SEED = 1508, 2071, 3000, 42


class Param:
    def __init__(self, epochs, n_user=N_USER, n_item=N_ITEM, batch=BATCH):
        self.n_user, self.n_item, self.k, self.lam = n_user, n_item, 16, 0.1
        self.seed, self.lr, self.lr_decay, self.momentum = SEED, 0.001, 0.95, 0.9
        self.epochs, self.batch = epochs, batch


def _arr3(triple):
    u, i, r = triple
    return np.stack([u.astype(np.float64), i.astype(np.float64), r / 5.0])


def test_scratch_train_vs_reference_golden(toy, cuda_dev):
    """Scratch.train (per-epoch baseTrain + baseTest) == the reference run: losses 1e-3 rel, final
    weights 1e-4 abs, test RMSE / HR 1e-3 rel."""
    from ultrare_b200.method.scratch import Scratch
    from ultrare_b200.method.utils import MF
    from ultrare_b200.read import RatingData, loadData
    z = load_gold("toy_train.npz")
    epochs = int(z["epochs"])
    P0, Q0 = init_weights(int(z["weight_seed"]))
    n = len(toy["train"][0])
    perms = [omf.feistel_perm(n, omf.perm_key(int(z["perm_seed"]), 0, ep)) for ep in range(epochs)]
    train = loadData(RatingData(_arr3(toy["train"])), BATCH, 1, True, perms=perms)
    test = loadData(RatingData(_arr3(toy["test"])), BATCH, 1, False)
    sc = Scratch(Param(epochs), 'mf')
    model = sc.train(train, test, [], 0, '', 0, MF.from_weights(P0, Q0))
    np.testing.assert_allclose(sc.log['train_loss'], z["losses"], rtol=1e-3)
    assert np.abs(model.user_mat.weight.cpu().numpy() - z["P_final"]).max() < 1e-4
    assert np.abs(model.item_mat.weight.cpu().numpy() - z["Q_final"]).max() < 1e-4
    assert abs(sc.log['test_rmse'][-1] - float(z["test_rmse"])) / float(z["test_rmse"]) < 1e-3
    assert abs(sc.log['test_hr'][-1] - float(z["test_hr"])) / float(z["test_hr"]) < 1e-3
    assert abs(sc.log['test_ndcg'][-1] - float(z["test_ndcg_ref"])) / float(z["test_ndcg_ref"]) < 2e-2   # tie rule, H7
    # inline Feistel permutation (no explicit perm): same result, the kernel regenerates the same order
    train2 = loadData(RatingData(_arr3(toy["train"])), BATCH, 1, True)
    sc2 = Scratch(Param(epochs), 'mf')
    sc2.seed = int(z["perm_seed"])
    sc2.train(train2, test, [], 0, '', 0, MF.from_weights(P0, Q0))
    np.testing.assert_allclose(sc2.log['train_loss'], z["losses"], rtol=1e-3)


def _sisa_inputs(toy, z, is_del, phase, K, epochs):
    from ultrare_b200.read import RatingData, loadData, readRating
    import pandas as pd
    groups0 = osisa.uniform_groups(N_USER, K)
    tr = pd.DataFrame({0: toy["train"][0], 1: toy["train"][1], 2: toy["train"][2]})
    te = pd.DataFrame({0: toy["test"][0], 1: toy["test"][1], 2: toy["test"][2]})
    trr, idx = readRating(tr, N_USER, 5, list(z["del_user"]) if is_del else [], [], K, groups0, 'a')
    ter, _ = readRating(te, N_USER, 5, [], [], K, idx)
    tl, sl = [], []
    for s in range(K):
        n = trr[s].shape[1]
        perms = [omf.feistel_perm(n, omf.perm_key(SEED + phase, s, ep)) for ep in range(epochs)]
        tl.append(loadData(RatingData(trr[s]), BATCH, 1, True, perms=perms))
        sl.append(loadData(RatingData(ter[s]), BATCH, 1, False))
    total = loadData(RatingData(np.hstack(ter)), BATCH, 1, False)
    return tl, sl, total, idx, trr


def _make_sisa(K, idx, epochs, mode):
    from ultrare_b200.method.sisa import Sisa
    from ultrare_b200.method.utils import MF

    class InjectedSisa(Sisa):
        def _new_model(self, id, user_rows=None):
            P0, Q0 = init_weights(100 + id - 1)
            if user_rows is not None:
                P0 = P0[user_rows.cpu().numpy()]
            return MF.from_weights(P0, Q0)

    s = InjectedSisa(Param(epochs), 'mf', K, idx)
    s.epoch_eval = mode
    return s


def test_sisa_learn_unlearn_faithful_vs_reference_golden(toy, cuda_dev, tmp_path):
    """The whole SISA path vs the reference's own Sisa.learn / Sisa.unlearn on toy data (K=3, 2 epochs):
    shard membership bit-exact, retrain_gid bit-exact, merged/item tables 1e-4, log0 RMSE/HR 1e-3,
    and the per-epoch logs incl. the model_list+[model] quirk (scratch.py:83-97)."""
    z = load_gold("toy_sisa.npz")
    K, epochs = int(z["K"]), int(z["epochs"])
    tl, sl, total, idx, trr = _sisa_inputs(toy, z, False, 0, K, epochs)
    for s in range(K):
        assert np.array_equal(np.asarray(idx[s]), z[f"group{s}"]) and trr[s].shape[1] == int(z[f"learn_train_n{s}"])
    sisa = _make_sisa(K, idx, epochs, 'faithful')
    d1 = str(tmp_path / "learn")
    os.makedirs(d1)
    models = sisa.learn(tl, sl, total, 0, d1)
    assert np.abs(models[0].user_mat.weight.cpu().numpy() - z["learn_merged"]).max() < 1e-4
    for s in range(K):
        assert np.abs(models[s].item_mat.weight.cpu().numpy() - z[f"learn_Q{s}"]).max() < 1e-4
        assert models[s].user_mat.weight is models[0].user_mat.weight
    ref0 = z["learn_log0"]
    got0 = np.load(d1 + "/log0.npy", allow_pickle=True).item()
    assert abs(got0['total_rmse'] - ref0[0]) / ref0[0] < 1e-3
    assert abs(got0['total_hr'] - ref0[2]) / ref0[2] < 1e-3
    assert abs(got0['total_ndcg'] - ref0[1]) / ref0[1] < 2e-2
    np.testing.assert_allclose(sisa.log['train_loss'], z["learn_log_train_loss"], rtol=1e-3)
    for key in ('test_rmse', 'total_rmse', 'test_hr', 'total_hr'):
        np.testing.assert_allclose(sisa.log[key], z["learn_log_" + key], rtol=1e-3, err_msg=key)
    for key in ('test_ndcg', 'total_ndcg'):
        np.testing.assert_allclose(sisa.log[key], z["learn_log_" + key], rtol=3e-2, err_msg=key)
    for s in range(K):     # artefact names / shapes of scratch.py:131-144
        assert np.load(d1 + f"/user_mat{s+1}.npy").shape == (N_USER, 16)
        assert np.load(d1 + f"/item_mat{s+1}.npy").shape == (N_ITEM, 16)
        assert os.path.exists(d1 + f"/model{s+1}.pth") and os.path.exists(d1 + f"/log{s+1}.npy")
        # log{i}.npy is saved as shard i finishes (scratch.py:144): the accumulated entries of shards 1..i only
        lg = np.load(d1 + f"/log{s+1}.npy", allow_pickle=True).item()
        assert all(len(v) == (s + 1) * epochs for v in lg.values()), {k: len(v) for k, v in lg.items()}
        np.testing.assert_allclose(lg['train_loss'], z["learn_log_train_loss"][:(s + 1) * epochs], rtol=1e-3)
        np.testing.assert_allclose(lg['total_rmse'], z["learn_log_total_rmse"][:(s + 1) * epochs], rtol=1e-3)

    # ---- unlearn
    tl, sl, total, idx2, trr = _sisa_inputs(toy, z, True, 1, K, epochs)
    for s in range(K):
        assert trr[s].shape[1] == int(z[f"unlearn_train_n{s}"])
    sisa2 = _make_sisa(K, idx2, epochs, 'faithful')
    models2 = sisa2.unlearn(models, tl, sl, total, list(z["del_user"]), 0, '')
    assert sorted(sisa2.retrain_gid) == z["retrain_gid"].tolist()
    assert np.abs(models2[0].user_mat.weight.cpu().numpy() - z["unlearn_merged"]).max() < 1e-4
    for s in range(K):
        assert np.abs(models2[s].item_mat.weight.cpu().numpy() - z[f"unlearn_Q{s}"]).max() < 1e-4
    ref0 = z["unlearn_log0"]
    assert abs(sisa2.final_log['total_rmse'] - ref0[0]) / ref0[0] < 1e-3
    assert abs(sisa2.final_log['total_hr'] - ref0[2]) / ref0[2] < 1e-3
    np.testing.assert_allclose(sisa2.log['train_loss'], z["unlearn_log_train_loss"], rtol=1e-3)


def test_sisa_compact_tables_equal_full_tables(toy, cuda_dev):
    """epoch_eval='none' (compact per-shard user tables) gives the reference's merged table / item
    tables / log0 too: rows a shard does not own never matter after the merge."""
    z = load_gold("toy_sisa.npz")
    K, epochs = int(z["K"]), int(z["epochs"])
    tl, sl, total, idx, _ = _sisa_inputs(toy, z, False, 0, K, epochs)
    sisa = _make_sisa(K, idx, epochs, 'none')
    models = sisa.learn(tl, sl, total, 0, '')
    assert np.abs(models[0].user_mat.weight.cpu().numpy() - z["learn_merged"]).max() < 1e-4
    for s in range(K):
        assert np.abs(models[s].item_mat.weight.cpu().numpy() - z[f"learn_Q{s}"]).max() < 1e-4
    assert abs(sisa.final_log['total_rmse'] - z["learn_log0"][0]) / z["learn_log0"][0] < 1e-3
    np.testing.assert_allclose(sisa.log['train_loss'], z["learn_log_train_loss"], rtol=1e-3)
    tl, sl, total, idx2, _ = _sisa_inputs(toy, z, True, 1, K, epochs)
    sisa2 = _make_sisa(K, idx2, epochs, 'final')
    models2 = sisa2.unlearn(models, tl, sl, total, list(z["del_user"]), 0, '')
    assert sorted(sisa2.retrain_gid) == z["retrain_gid"].tolist()
    assert np.abs(models2[0].user_mat.weight.cpu().numpy() - z["unlearn_merged"]).max() < 1e-4
    assert abs(sisa2.final_log['total_rmse'] - z["unlearn_log0"][0]) / z["unlearn_log0"][0] < 1e-3


def test_ot_cluster_vs_oracle_and_reference(cuda_dev):
    """GPU ot_cluster (Sinkhorn potentials + balanced rounding) against
    (a) the same outer loop with the float64 Sinkhorn oracle + the oracle's rounding as plan solver;
    (b) the exact-EMD labels of one outer iteration (what the reference's ot.emd gives): equal up to cost ties;
    (c) the reference's own full ot_cluster run (golden, exact LP in place of POT): group sizes exactly n/k as the
        reference's, label agreement reported and gated at >= 0.98 (H1)."""
    from ultrare_b200.method.utils import SINKHORN_SCHEDULE, ot_cluster, ot_cluster_device
    z = load_gold("ot_cluster.npz")
    X, k = z["X"], int(z["k"])
    n = len(X)

    def sinkhorn_rounded_plan(a, b, M):
        M = np.asarray(M, dtype=np.float64)
        scale = M.min(axis=1).mean()
        g = oot.sinkhorn_log(M, [(e * scale, i) for e, i in SINKHORN_SCHEDULE])[2]
        lab, _ = oot.balance_labels(M.astype(np.float32), np.argmax(g[None, :] - M, axis=1))
        return np.eye(M.shape[1])[lab]                       # one-hot rows: assign() recovers the labels

    np.random.seed(int(z["np_seed"]))
    in_o, lab_o, cen_o, it_o = oot.ot_cluster(X, k, plan_fn=sinkhorn_rounded_plan)
    np.random.seed(int(z["np_seed"]))
    c_init = X[np.random.choice(n, size=k, replace=False)]
    in_f, lab_f, _, _ = ot_cluster_device(X, k, centroid0=c_init, tol=0.0, warm_start=False)   # the fixed schedule
    assert (lab_f == lab_o).mean() >= 0.995
    assert abs(float(in_f) - float(in_o)) / float(in_o) < 1e-4
    np.random.seed(int(z["np_seed"]))
    inertia, label = ot_cluster(X, k)            # product default: warm start + early exit
    assert label.dtype == np.int64 and label.shape == (n,)
    assert (label == lab_o).mean() >= 0.99
    assert abs(float(inertia) - float(in_o)) / float(in_o) < 1e-3
    # (b) first outer iteration against exact EMD
    np.random.seed(int(z["np_seed"]))
    c0 = X[np.random.choice(n, size=k, replace=False)]
    _, lab1, _, _ = ot_cluster_device(X, k, max_iters=1, centroid0=c0)
    G = oot.emd_lp(np.ones(n) / n, np.ones(k) / k, oot.cost_matrix_ref_fp32(X, c0).T)
    assert (lab1 == oot.assign(G)).mean() >= 0.998
    # (c) the reference's full run
    agree = (label == z["label"]).mean()
    sizes = np.bincount(label, minlength=k)
    print(f"ot_cluster vs reference EMD run: label agreement {agree:.4f}, sizes {sizes.tolist()}, "
          f"inertia {float(inertia):.3f} vs {float(z['inertia']):.3f}")
    assert sizes.tolist() == np.bincount(z["label"], minlength=k).tolist() == [n // k] * k
    assert agree >= 0.98
    assert abs(float(inertia) - float(z["inertia"])) / float(z["inertia"]) < 1e-3


def test_ot_cluster_warm_start_on_the_input_that_degenerated_in_round_1(cuda_dev):
    """The real failing input of round 1 (profiles/r1_notes.md): synthetic ml1m, the user table after two epochs of
    full training (`main.py --synth --epoch 2 --group 0`), centroid start users [2680, 1199, 926, 4420, 1670]
    (Appendix C).  Outer iteration 2, warm-started at the small eps, used to put all 6040 users on one centroid.
    No host-side guard exists any more: the log-domain column sums must carry it, with warm_start=True."""
    from ultrare_b200 import synth
    from ultrare_b200.method.scratch import Scratch
    from ultrare_b200.method.utils import ot_cluster_device
    from ultrare_b200.read import RatingData, loadData
    train, test = synth.ml_like()
    U, I = synth.ML1M["n_user"], synth.ML1M["n_item"]

    class P:
        n_user, n_item, k, lam, seed, lr, lr_decay, momentum, epochs, batch = U, I, 16, 0.1, 42, 1e-3, 0.95, 0.9, 2, 30000

    tr = np.stack([train[0].astype(np.float64), train[1].astype(np.float64), train[2] / 5.0])
    te = np.stack([test[0].astype(np.float64), test[1].astype(np.float64), test[2] / 5.0])
    model = Scratch(P, 'mf').train(loadData(RatingData(tr), 30000, 1), loadData(RatingData(te), 30000, 1, False),
                                   [], 0, '', 0)
    emb = model.user_mat.weight.detach().cpu().numpy()
    start = [2680, 1199, 926, 4420, 1670]
    inertia, label, cen, it = ot_cluster_device(emb, 5, centroid0=emb[start], warm_start=True)
    sizes = np.bincount(label, minlength=5)
    assert sizes.tolist() == [1208] * 5, sizes
    assert np.isfinite(cen).all() and np.isfinite(inertia) and it >= 2
    # the same start without the warm start ends in the same kind of grouping (same sizes, close inertia)
    inertia_c, label_c, _, _ = ot_cluster_device(emb, 5, centroid0=emb[start], warm_start=False)
    assert np.bincount(label_c, minlength=5).tolist() == [1208] * 5
    assert abs(float(inertia) - float(inertia_c)) / float(inertia_c) < 2e-2


def test_instance_run_full_then_group_end_to_end(toy, cuda_dev, tmp_path, monkeypatch):
    """main.py's dispatch on the toy dataset: runFull (group=0) then runGroup (emb-ot, sisa), checking the
    artefact names / keys the reference writes (config.py:60-77, scratch.py:131-144, sisa.py:18-23)."""
    import ultrare_b200.config as cfg
    import ultrare_b200.group as grp
    from ultrare_b200 import synth
    data, save = str(tmp_path / "data"), str(tmp_path / "result")
    for mod in (cfg, grp):
        monkeypatch.setattr(mod, "DATA_DIR", data)
        monkeypatch.setattr(mod, "SAVE_DIR", save)
    synth.ensure_dataset("toy")
    p0 = cfg.InsParam("toy", 2, 1, [32], 0, 2, "rand")
    assert np.array_equal(p0.del_user, osisa.deletion_set(N_USER, 2))
    cfg.Instance(p0).runFull(is_save=True, verbose=0)
    base = save + "/2/rand/toy_g0"
    for sub in ("MF_full_train", "MF_retrain"):
        for f in ("model0.pth", "user_mat0.npy", "item_mat0.npy", "log0.npy"):
            assert os.path.exists(f"{base}/{sub}/{f}"), (sub, f)
    log = np.load(base + "/MF_full_train/log0.npy", allow_pickle=True).item()
    assert len(log['train_loss']) == 2 and log['train_loss'][1] < log['train_loss'][0]
    assert os.path.exists(base + "/param.pkl") and os.path.exists(base + "/deletion.npy")

    p3 = cfg.InsParam("toy", 2, 1, [32], 3, 2, "rand")
    ins = cfg.Instance(p3)
    ins.runGroup(is_save=True, learn_type='sisa', group_type='emb-ot', n_group=3, verbose=0)
    gdir = save + "/2/rand/toy_g3"
    for sub in ("MF_emb-ot_sisa_learn", "MF_emb-ot_sisa_unlearn"):
        l0 = np.load(f"{gdir}/{sub}/log0.npy", allow_pickle=True).item()
        assert set(l0) == {'total_rmse', 'total_ndcg', 'total_hr'} and np.isfinite(l0['total_rmse'])
    cache = np.load(data + "/toy/val/emb-ot3.npy", allow_pickle=True)
    sizes = sorted(len(g) for g in cache)
    assert sum(sizes) == N_USER and sizes[-1] - sizes[0] <= 0.05 * N_USER
    # routing against the brute-force restatement of sisa.py:76-81
    sisa = ins.last_sisa
    assert sisa.retrain_gid == osisa.route_deletions(sisa.group_index, p3.del_user)


def test_instance_run_group_uniform_delper5(toy, cuda_dev, tmp_path, monkeypatch):
    """The other branches reachable from the CLI (SURVEY.md §8 f4): group_type='uniform' (runGroup's default,
    config.py:190, groups of read.py:21-33) and --delper 5: artefacts, routing, and the deletion set of Appendix C."""
    import ultrare_b200.config as cfg
    import ultrare_b200.group as grp
    from ultrare_b200 import synth
    data, save = str(tmp_path / "data"), str(tmp_path / "result")
    for mod in (cfg, grp):
        monkeypatch.setattr(mod, "DATA_DIR", data)
        monkeypatch.setattr(mod, "SAVE_DIR", save)
    synth.ensure_dataset("toy")
    p = cfg.InsParam("toy", 2, 1, [32], 4, 5, "rand")
    assert np.array_equal(p.del_user, osisa.deletion_set(N_USER, 5)) and len(p.del_user) == int(0.05 * N_USER)
    ins = cfg.Instance(p)
    ins.runGroup(is_save=True, learn_type='sisa', group_type='uniform', n_group=4, verbose=0)
    gdir = save + "/5/rand/toy_g4"
    for sub in ("MF_uniform_sisa_learn", "MF_uniform_sisa_unlearn"):
        l0 = np.load(f"{gdir}/{sub}/log0.npy", allow_pickle=True).item()
        assert set(l0) == {'total_rmse', 'total_ndcg', 'total_hr'} and np.isfinite(l0['total_rmse'])
    sisa = ins.last_sisa
    groups = osisa.uniform_groups(N_USER, 4)
    assert sorted(map(sorted, sisa.group_index)) == sorted(map(sorted, groups))
    assert sisa.retrain_gid == osisa.route_deletions(sisa.group_index, p.del_user)


@pytest.mark.gpu
@pytest.mark.parametrize("n_group,with_del,sort", [(1, False, 'r'), (5, True, 'a'), (7, True, 'r')])
def test_read_rating_device_equals_host(n_group, with_del, sort):
    """readRatingDevice (partition kernel) == readRating (host filter, reference read.py:36-68): same groups, same
    rows in the same order, bit-equal float32 ratings; host views of the device-backed datasets equal too."""
    import pandas as pd
    from ultrare_b200 import kernels as kn
    from ultrare_b200.read import RatingData, readRating, readRatingDevice
    rng = np.random.default_rng(5)
    n_user, n_item, n = 700, 300, 60000
    df = pd.DataFrame({0: rng.integers(0, n_user, n), 1: rng.integers(0, n_item, n), 2: rng.integers(1, 6, n)})
    del_user = list(rng.choice(n_user, 40, replace=False)) if with_del else []
    host, gi_h = readRating(df, n_user, 5, del_user, [], n_group, [], sort)
    dev, gi_d, total = readRatingDevice(df, n_user, 5, del_user, [], n_group, [], sort, device='cuda')
    assert [list(g) for g in gi_h] == [list(g) for g in gi_d]
    for g in range(n_group):
        want = RatingData(host[g]).records('cuda').cpu().numpy()
        got = dev[g].records('cuda').cpu().numpy()
        assert got.shape == want.shape and np.array_equal(got, want), g
        assert np.array_equal(dev[g].users, host[g][0].astype(int)) and np.array_equal(dev[g].ratings, host[g][2])
        assert np.array_equal(dev[g]._raw, host[g])
    assert np.array_equal(total.records('cuda').cpu().numpy(),
                          RatingData(np.hstack(host)).records('cuda').cpu().numpy())
    # compact-row remap == the pack kernel's remap
    row_of = torch.from_numpy(rng.integers(0, 50, n_user).astype(np.int32)).cuda()
    g = n_group - 1
    assert np.array_equal(dev[g].records_mapped('cuda', row_of, 't').cpu().numpy(),
                          RatingData(host[g]).records_mapped('cuda', row_of, 't').cpu().numpy())


@pytest.mark.gpu
def test_read_rating_device_ragged_edges():
    """Users without ratings, an empty group, ids beyond n_user, a table smaller than one CTA tile."""
    import pandas as pd
    from ultrare_b200.read import RatingData, readRating, readRatingDevice
    from ultrare_b200 import kernels as kn
    df = pd.DataFrame({0: [3, 3, 9, 0, 12, 3, 9], 1: [1, 2, 3, 4, 5, 6, 7], 2: [5, 4, 3, 2, 1, 5, 4]})
    groups = [[0, 1], [2], [3, 9], [12]]
    # both table layouts, on a 3-row table where the shapes alone cannot tell them apart
    t3 = torch.tensor([[0., 1., 5.], [1., 2., 4.], [0., 3., 1.]], dtype=torch.float64, device='cuda')
    own = torch.tensor([1, 0], dtype=torch.int32, device='cuda')
    r_rows, o_rows = kn.partition_interactions(t3, 5, own, None, 2, columns=False)
    r_cols, o_cols = kn.partition_interactions(t3.t().contiguous(), 5, own, None, 2, columns=True)
    assert o_rows.tolist() == o_cols.tolist() == [0, 1, 3] and torch.equal(r_rows, r_cols)
    assert r_rows[:, :2].tolist() == [[1, 2], [0, 1], [0, 3]]
    host, _ = readRating(df, 10, 5, [9], [], 4, groups)
    dev, _, total = readRatingDevice(df, 10, 5, [9], [], 4, groups, device='cuda')
    assert [len(d) for d in dev] == [h.shape[1] for h in host] == [1, 0, 3, 1]
    for g in range(4):
        assert np.array_equal(dev[g].records('cuda').cpu().numpy(), RatingData(host[g]).records('cuda').cpu().numpy())
    assert len(total) == 5


@pytest.mark.gpu
def test_sisa_full_size_ml1m_unlearn_properties(cuda_dev):
    """BASELINE config 2 at full size (ml1m shape, K=5, 897 k interactions) through the public Sisa surface, checked
    by properties that do not need a full reference run: the retrain set equals the oracle's routing; shards outside
    it keep their item tables bit for bit and their owners keep their merged user rows; retrained shards change;
    the final ensemble metrics equal the CPU oracle's baseTest on the tables the GPU produced."""
    import pandas as pd
    from oracle import evalm as oev
    from ultrare_b200 import synth
    from ultrare_b200.method.sisa import Sisa
    from ultrare_b200.read import RatingData, loadData, readRating
    train, test = synth.ml_like()
    U, I, K, E, B = 6040, 3416, 5, 2, 30000
    tr = pd.DataFrame({0: train[0], 1: train[1], 2: train[2]})
    te = pd.DataFrame({0: test[0], 1: test[1], 2: test[2]})
    trr, groups = readRating(tr, U, 5, [], [], K, [], 'a')
    ter, _ = readRating(te, U, 5, [], [], K, groups)
    del_user = [int(x) for x in groups[1][:7]] + [int(x) for x in groups[3][5:9]]      # shards 1 and 3 only
    trd, _ = readRating(tr, U, 5, del_user, [], K, groups, 'r')
    assert sum(a.shape[1] for a in trr) == len(train[0]) > 890_000

    class P:
        n_user, n_item, k, lam, seed, lr, lr_decay, momentum, epochs, batch = U, I, 16, 0.1, 42, 0.001, 0.95, 0.9, E, B

    def loaders(arrs, shuffle):
        return [loadData(RatingData(a), B, 1, shuffle) for a in arrs]

    test_dl = loaders(ter, False)
    test_total = np.hstack(ter)
    test_data = loadData(RatingData(test_total), B, 1, False)
    s1 = Sisa(P, 'mf', K, groups)
    s1.epoch_eval = 'none'
    before = s1.learn(loaders(trr, True), test_dl, test_data, 0, '')
    P_before = before[0].user_mat.weight.data.clone()
    Q_before = [m.item_mat.weight.data.clone() for m in before]
    log_learn = dict(s1.final_log)

    s2 = Sisa(P, 'mf', K, groups)
    s2.epoch_eval = 'none'
    after = s2.unlearn(before, loaders(trd, True), test_dl, test_data, del_user, 0, '')
    assert s2.retrain_gid == set(osisa.route_deletions(groups, del_user)) == {1, 3}
    # both routing paths (host look-ups for a small deletion set, the owner-map kernel for a large one) give the
    # same flags, with out-of-range and unowned ids ignored
    s3 = Sisa(P, 'mf', K, groups)
    odd = list(del_user) + [-5, 10 ** 9]
    f_host = s3.route(odd).cpu().numpy()
    s3.ROUTE_ON_HOST_MAX = 0
    f_dev = s3.route([u for u in odd if 0 <= u < s3.n_user]).cpu().numpy()
    assert np.array_equal(f_host, f_dev) and set(np.flatnonzero(f_host)) == {1, 3}
    P_after = after[0].user_mat.weight.data
    for g in range(K):
        Qg = after[g].item_mat.weight.data
        rows = torch.as_tensor(np.asarray(groups[g]), device=P_after.device)
        if g in s2.retrain_gid:
            assert not torch.equal(Qg, Q_before[g])
            assert not torch.equal(P_after[rows], P_before[rows])
        else:
            assert torch.equal(Qg, Q_before[g])
            assert torch.equal(P_after[rows], P_before[rows])
    assert len(s2.log['train_loss']) == 2 * E and all(np.isfinite(s2.log['train_loss']))
    # fresh N(0,1) tables on nearly the same data: the first-epoch loss of shard 1 stays in the same range
    assert abs(s2.log['train_loss'][0] - s1.log['train_loss'][E]) < 0.1 * s1.log['train_loss'][E]

    # final metrics (sisa.py:18-23 -> baseTest) against the oracle on the GPU's own tables
    Pm = P_after.cpu().numpy()
    Qs = [m.item_mat.weight.data.cpu().numpy() for m in after]
    tu, ti, trt = test_total[0].astype(np.int64), test_total[1].astype(np.int64), test_total[2].astype(np.float32)
    rmse, ndcg, hr, _ = oev.base_test([Pm] * K, Qs, tu, ti, trt)
    got = s2.final_log
    assert abs(got['total_rmse'] - rmse) < 1e-4 * rmse
    assert abs(got['total_ndcg'] - ndcg) < 1e-4 and abs(got['total_hr'] - hr) < 1e-4
    assert got['total_rmse'] != log_learn['total_rmse']


@pytest.mark.gpu
def test_instance_read_data_device_equals_host_branch(toy, cuda_dev, tmp_path, monkeypatch):
    """Instance._read_data: the device ingest (default) and the host split (URE_HOST_INGEST=1) give the same group
    order and bit-equal records per group, for the deletion-filtered training read and the test read."""
    import ultrare_b200.config as cfg
    import ultrare_b200.group as grp
    from ultrare_b200 import synth
    data, save = str(tmp_path / "data"), str(tmp_path / "result")
    for mod in (cfg, grp):
        monkeypatch.setattr(mod, "DATA_DIR", data)
        monkeypatch.setattr(mod, "SAVE_DIR", save)
    synth.ensure_dataset("toy")
    ins = cfg.Instance(cfg.InsParam("toy", 2, 1, [32], 4, 2, "rand"))
    monkeypatch.setenv("URE_HOST_INGEST", "0")
    d_train, d_idx, d_test, d_total = ins._read_data(True, 4, [])
    monkeypatch.setenv("URE_HOST_INGEST", "1")
    h_train, h_idx, h_test, h_total = ins._read_data(True, 4, [])
    assert [list(g) for g in d_idx] == [list(g) for g in h_idx]
    for a, b in list(zip(d_train, h_train)) + list(zip(d_test, h_test)) + [(d_total, h_total)]:
        assert len(a) == len(b) > 0
        assert torch.equal(a.records(cuda_dev), b.records(cuda_dev))


@pytest.mark.gpu
def test_balanced_rounding_from_a_degenerate_assignment_is_still_the_exact_optimum(cuda_dev):
    """Whatever the potentials, the argmax assignment is cost-optimal for ITS group sizes -- even the degenerate one
    with every user in group 0 (what round 1's underflow produced).  The successive-shortest-path rounding therefore
    ends at the exact balanced optimum from there too: n*(k-1)/k augmentations, labels equal to the exact LP's."""
    from ultrare_b200 import kernels as kn
    rng = np.random.default_rng(5)
    n, k = 1000, 4
    X = rng.standard_normal((n, 16)).astype(np.float32)
    M = kn.cost_matrix(torch.tensor(X, device=cuda_dev), torch.tensor(X[:k].copy(), device=cuda_dev))
    g = torch.tensor([1e6, 0.0, 0.0, 0.0], device=cuda_dev)           # potentials that send every user to group 0
    label, _, cnt = kn.assign_centroids(M, k, g, None)
    assert cnt.cpu().numpy().tolist() == [n, 0, 0, 0]
    status = kn.balance_labels(M, k, label, cnt).cpu().numpy()
    assert status.tolist() == [n - n // k, 0, 0] and cnt.cpu().numpy().tolist() == [n // k] * k
    Mh = M.cpu().numpy()[:, :k]
    emd = oot.assign(oot.emd_lp(np.ones(n) / n, np.ones(k) / k, Mh))
    assert (label.cpu().numpy() == emd).mean() >= 0.998


@pytest.mark.gpu
def test_optimistic_owner_launch_hit_and_miss(cuda_dev):
    """Sisa.unlearn without artefacts queues the owner launch with the capacities of the last plan of the same shapes
    (kernels._PLAN_HINTS) instead of waiting for the plan read-back; the kernels verify them on the device
    (hparams.owner_plan).  A hit reproduces the waited-for pass bit for bit; a remembered plan that does not cover
    the batch trains nothing, raises PlanHintMiss when the deferred losses are read, and the pass is repeated."""
    import pandas as pd
    from ultrare_b200 import kernels as kn, synth
    from ultrare_b200.method.sisa import Sisa
    from ultrare_b200.read import RatingData, loadData, readRating
    train, test = synth.ml_like()
    U, I, K, E, B = 6040, 3416, 5, 2, 30000
    tr = pd.DataFrame({0: train[0], 1: train[1], 2: train[2]})
    te = pd.DataFrame({0: test[0], 1: test[1], 2: test[2]})
    trr, groups = readRating(tr, U, 5, [], [], K, [], 'a')
    ter, _ = readRating(te, U, 5, [], [], K, groups)
    del_user = [int(g[0]) for g in groups]                                   # every shard retrains
    trd, _ = readRating(tr, U, 5, del_user, [], K, groups, 'r')

    class P:
        n_user, n_item, k, lam, seed, lr, lr_decay, momentum, epochs, batch = U, I, 16, 0.1, 42, 0.001, 0.95, 0.9, E, B

    mk = lambda arrs, sh: [loadData(RatingData(a), B, 1, sh) for a in arrs]
    tdl = mk(ter, False)
    tdata = loadData(RatingData(np.hstack(ter)), B, 1, False)

    def new():
        s = Sisa(P, 'mf', K, groups)
        s.epoch_eval = 'none'
        return s

    models = new().learn(mk(trr, True), tdl, tdata, 0, '')
    train_dl = mk(trd, True)
    kn._PLAN_HINTS.clear()                                                   # (learn remembers its plan as well)

    def run():
        un = new()
        out = un.unlearn(models, train_dl, tdl, tdata, del_user, 0, '')
        return un, [m.item_mat.weight.data.clone() for m in out], out[0].user_mat.weight.data.clone()

    un0, q0, p0 = run()                                                      # waits for its plan, remembers it
    assert not un0._last_batch.optimistic and len(kn._PLAN_HINTS) >= 1
    un1, q1, p1 = run()                                                      # queued on the remembered plan
    assert un1._last_batch.optimistic and un1._last_batch.owner_plan['optimistic']
    assert torch.equal(p0, p1) and all(torch.equal(a, b) for a, b in zip(q0, q1))
    same_log = lambda a, b: all(abs(a[k] - b[k]) <= 1e-12 for k in a)           # metric sums: fp64 atomics, any order
    assert same_log(un1.final_log, un0.final_log)
    sig = un1._last_batch._plan_sig
    good = kn._PLAN_HINTS[sig]
    kn._PLAN_HINTS[sig] = (max(1, good[0] // 2), max(16, good[1] // 2), good[2], good[3])   # too small: must miss
    un2, q2, p2 = run()
    assert not un2._last_batch.optimistic                                    # the repeat waited for the real plan
    assert kn._PLAN_HINTS[sig] == good
    assert torch.equal(p0, p2) and all(torch.equal(a, b) for a, b in zip(q0, q2))
    assert same_log(un2.final_log, un0.final_log)


@pytest.mark.gpu
def test_eager_upload_from_the_constructor(cuda_dev):
    """read.EAGER_UPLOAD_DEVICE: a RatingData built on a page-locked float64 [3, n] array starts its host -> device copy
    in the constructor (side stream); records(), records_mapped() and upload_many() then pack from the device columns.
    Same records as the ordinary upload; arrays that do not qualify (small, pageable) take the ordinary way."""
    from ultrare_b200 import kernels as kn, read as rd
    from ultrare_b200.read import RatingData
    rng = np.random.default_rng(4)
    n, U, I = 200_000, 5000, 3000
    raw = np.stack([rng.integers(0, U, n), rng.integers(0, I, n), rng.integers(1, 6, n) / 5.0]).astype(np.float64)
    row_of = torch.tensor(rng.permutation(U).astype(np.int32), device=cuda_dev)
    want = RatingData(raw).records(cuda_dev).cpu()
    want_m = RatingData(raw).records_mapped(cuda_dev, row_of, 't').cpu()
    pinned, small = kn.pinned_copy(raw), kn.pinned_copy(raw[:, :1000].copy())
    rd.EAGER_UPLOAD_DEVICE = cuda_dev
    try:
        a, b, c, d_, e = RatingData(pinned), RatingData(pinned), RatingData(pinned), RatingData(small), RatingData(raw)
        assert a._eager is not None and b._eager is not None and d_._eager is None and e._eager is None
        assert torch.equal(a.records(cuda_dev).cpu(), want) and a._eager is None
        assert torch.equal(b.records_mapped(cuda_dev, row_of, 't').cpu(), want_m)
        RatingData.upload_many([c, d_, e], cuda_dev, row_of, 't')
        assert torch.equal(c.records_mapped(cuda_dev, row_of, 't').cpu(), want_m)
        assert torch.equal(e.records_mapped(cuda_dev, row_of, 't').cpu(), want_m)
        assert torch.equal(d_.records_mapped(cuda_dev, row_of, 't').cpu(), want_m[:1000])
    finally:
        rd.EAGER_UPLOAD_DEVICE = None
