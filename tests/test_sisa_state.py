"""Saved SISA states and deletion requests applied to them in a later run (Sisa.save_state / load_state /
apply_request, main.py --save-state / --unlearn-from).

CPU: request files, request validation, the effective request (request minus ledger), the manifest refusals, the
request run's flag checks.  GPU: save + load round trips bit-equal to the in-memory model; an unlearn from a loaded
state bit-equal to the in-process unlearn; two requests across a save / load equal to the in-process sequence; states
saved at 2 ranks loaded at 1 and 3 (threads); the CLI end to end in separate processes.  Before every load the module
caches a fresh process would not have are cleared (_fresh)."""
import json
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from oracle import sisa as osisa

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K_TOY = 3


def _fresh():
    from ultrare_b200 import kernels as kn
    from ultrare_b200.method import sisa
    sisa._OWNER_CACHE.clear()
    sisa._EVAL_ROWS.clear()
    kn._PLAN_HINTS.clear()


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
    """A hand-written manifest of a state of the toy source (no arrays)."""
    from ultrare_b200.method import sisa_state as st
    size, sha = st.file_digest(src['train_file'])
    man = dict(format=st.FORMAT_VERSION, K=K_TOY, slices=4, k=16, n_user=1508, n_item=2071, epochs=2, batch=3000,
               lr=0.001, lr_decay=0.95, lam=0.1, momentum=0.9, seed=42, combine='mean', epoch_eval='final',
               dataset='toy', grouping='uniform', max_rating=5,
               train_file=dict(path=src['train_file'], bytes=size, sha256=sha), test_file=src['test_file'], requests=0)
    man.update(over)
    d = tmp_path / "state"
    d.mkdir(exist_ok=True)
    (d / "manifest.json").write_text(json.dumps(man))
    return str(d), man


# ------------------------------------------------------------------------------------------------------------ CPU
def test_request_files_npy_text_and_csv(tmp_path):
    from ultrare_b200.method.sisa_state import parse_request_file
    np.save(tmp_path / "u.npy", np.array([5, 3, 9]))
    np.save(tmp_path / "p.npy", np.array([[1, 2], [3, 4]], dtype=np.int32))
    (tmp_path / "u.txt").write_text("5\n3\n\n# a comment\n9\n")
    (tmp_path / "p.csv").write_text("1,2\n3, 4\n")
    (tmp_path / "p.txt").write_text("1 2\n3\t4\n")
    (tmp_path / "empty.txt").write_text("")
    for name in ("u.npy", "u.txt"):
        got = parse_request_file(str(tmp_path / name), 'users')
        assert got.dtype == np.int64 and got.tolist() == [5, 3, 9]
    for name in ("p.npy", "p.csv", "p.txt"):
        got = parse_request_file(str(tmp_path / name), 'ratings')
        assert got.dtype == np.int64 and got.tolist() == [[1, 2], [3, 4]]
    assert parse_request_file(str(tmp_path / "empty.txt"), 'users').shape == (0,)
    assert parse_request_file(str(tmp_path / "empty.txt"), 'ratings').shape == (0, 2)
    with pytest.raises(ValueError, match="one id per line"):
        parse_request_file(str(tmp_path / "p.csv"), 'users')
    (tmp_path / "f.txt").write_text("1.5\n")
    with pytest.raises(ValueError, match="integers"):
        parse_request_file(str(tmp_path / "f.txt"), 'users')
    np.save(tmp_path / "obj.npy", np.array([1, None], dtype=object), allow_pickle=True)
    with pytest.raises(ValueError):
        parse_request_file(str(tmp_path / "obj.npy"), 'users')          # no pickle is ever loaded


def test_request_validation_errors():
    from ultrare_b200.method.sisa_state import validate_request
    u, p = validate_request([7, 3, 7], [[4, 1], [2, 0], [4, 1]], 10, 5)
    assert u.tolist() == [3, 7] and p.tolist() == [[2, 0], [4, 1]]
    u, p = validate_request([], [], 10, 5)
    assert u.shape == (0,) and p.shape == (0, 2)
    bad = [([-1], []), ([], [[-1, 0]]), ([], [[0, -2]]), ([10], []), ([], [[10, 0]]), ([], [[0, 5]]),
           ([], [[1, 2, 3]]), ([], [1, 2]), ([1.5], []), ([], [[0.5, 1]])]
    for users, pairs in bad:
        with pytest.raises(ValueError):
            validate_request(users, pairs, 10, 5)


def test_effective_request_is_the_request_minus_the_ledger():
    from ultrare_b200.method.sisa_state import deletion_table, effective_request, ledger_union, validate_request
    led_u, led_p = np.array([2, 5], dtype=np.int64), np.array([[1, 1], [3, 7]], dtype=np.int64)
    u, p = validate_request([5, 6, 2, 8], [[3, 7], [5, 0], [1, 2], [6, 3], [1, 1], [2, 9]], 10, 10)
    eu, ep = effective_request(u, p, led_u, led_p)
    # users 2 and 5 already deleted; pair (3, 7) and (1, 1) already deleted; (5, 0) and (2, 9) belong to deleted users
    assert eu.tolist() == [6, 8] and ep.tolist() == [[1, 2], [6, 3]]
    nu, np_ = ledger_union(led_u, led_p, eu, ep)
    assert nu.tolist() == [2, 5, 6, 8] and np_.tolist() == [[1, 1], [1, 2], [3, 7], [6, 3]]
    e2 = effective_request(u, p, nu, np_)
    assert len(e2[0]) == 0 and len(e2[1]) == 0
    e3 = effective_request(u, p, np.zeros(0, np.int64), np.zeros((0, 2), np.int64))
    assert e3[0].tolist() == u.tolist() and e3[1].tolist() == p.tolist()
    assert deletion_table(eu, ep).tolist() == [[6, -1], [8, -1], [1, 2], [6, 3]]


def test_manifest_refusals(tmp_path, monkeypatch):
    """load_state refuses a directory without a manifest, an incomplete one, another format version and a changed
    training file; the retained-data read refuses a train_index the reader does not return."""
    from ultrare_b200.method import sisa_state as st
    from ultrare_b200.method.sisa import Sisa
    src = _toy_source(tmp_path)
    empty = tmp_path / "nothing"
    empty.mkdir()
    with pytest.raises(ValueError, match="no manifest.json"):
        Sisa.load_state(str(empty))
    d, man = _manifest(tmp_path, src)
    (tmp_path / "state" / "manifest.json").write_text("{\"format\": 1, \"K\"")
    with pytest.raises(ValueError, match="JSON"):
        Sisa.load_state(d)
    for key in ('requests', 'train_file', 'slices'):
        _manifest(tmp_path, src, **{key: None})
        m = json.loads((tmp_path / "state" / "manifest.json").read_text())
        del m[key]
        (tmp_path / "state" / "manifest.json").write_text(json.dumps(m))
        with pytest.raises(ValueError, match="incomplete"):
            Sisa.load_state(d)
    _manifest(tmp_path, src, format=st.FORMAT_VERSION + 1)
    with pytest.raises(ValueError, match="format version"):
        Sisa.load_state(d)
    _manifest(tmp_path, src)
    with pytest.raises(ValueError, match="group_index_ids.npy is missing"):
        Sisa.load_state(d)                              # the manifest passes; the arrays are not there
    with open(src['train_file'], 'a') as f:             # one more rating: same path, other bytes
        f.write("0,0,5.0\n")
    with pytest.raises(ValueError, match="changed"):
        Sisa.load_state(d)
    # train_index: the count-sorted grouping the reader returns must be the stored one
    src = _toy_source(tmp_path)
    monkeypatch.setenv('URE_HOST_INGEST', '1')
    _, _, _, idx = st.read_retained(src, 1508, K_TOY, 1, 3000, [], [])
    st.check_train_index(idx, [list(g) for g in idx])
    with pytest.raises(ValueError, match="train_index"):
        st.check_train_index(idx, [idx[1], idx[0], idx[2]])
    with pytest.raises(ValueError, match="train_index"):
        st.check_train_index(idx, [idx[0][1:] + idx[0][:1], idx[1], idx[2]])


def test_request_run_flags(tmp_path):
    from ultrare_b200.main import _checked, main, parser
    for bad in (['--unlearn-from', 'd'], ['--unlearn-from', 'd', '--out', 'o'],
                ['--unlearn-from', 'd', '--forget-users', 'f'], ['--out', 'o'], ['--forget-ratings', 'f']):
        with pytest.raises(AssertionError):
            _checked(parser.parse_args(bad))
    a = _checked(parser.parse_args(['--unlearn-from', 'd', '--out', 'o', '--forget-ratings', 'f']))
    assert a.unlearn_from == 'd' and a.forget_users is None
    assert _checked(parser.parse_args(['--save-state'])).save_state
    src = _toy_source(tmp_path)
    d, _ = _manifest(tmp_path, src)
    (tmp_path / "u.txt").write_text("3\n")
    req = ['--unlearn-from', d, '--out', str(tmp_path / "out"), '--forget-users', str(tmp_path / "u.txt")]
    for extra, flag in ((['--slices', '2'], '--slices'), (['--group', '5'], '--group'), (['--epoch', '3'], '--epoch'),
                        (['--dataset', 'ml1m'], '--dataset'), (['--combine', 'fit'], '--combine'),
                        (['--grouping', 'rating-ot'], '--grouping'), (['--epoch-eval', 'none'], '--epoch-eval'),
                        (['--deltype', 'inter'], '--deltype'), (['--delper', '2'], '--delper'),
                        (['--save-state'], '--save-state')):
        with pytest.raises(AssertionError, match=flag):
            main(req + extra)
    out = tmp_path / "out"
    out.mkdir()
    (out / "x").write_text("")
    with pytest.raises(ValueError, match="not empty"):
        main(req + ['--slices', '4', '--group', '3', '--dataset', 'toy'])       # agreeing flags pass the check
    (tmp_path / "file").write_text("")
    with pytest.raises(ValueError, match="not empty"):
        main(req[:2] + ['--out', str(tmp_path / "file")] + req[4:])


# ------------------------------------------------------------------------------------------------------------ GPU
class _Param:
    def __init__(self, epochs, n_user=1508, n_item=2071):
        self.n_user, self.n_item, self.k, self.lam = n_user, n_item, 16, 0.1
        self.seed, self.lr, self.lr_decay, self.momentum = 42, 0.001, 0.95, 0.9
        self.epochs, self.batch = epochs, 3000


def _read(src, K, R, users=(), pairs=()):
    from ultrare_b200.method import sisa_state as st
    tl, sl, total, idx = st.read_retained(src, 1508, K, R, 3000, np.asarray(users, dtype=np.int64),
                                          np.asarray(pairs, dtype=np.int64).reshape(-1, 2))
    return tl, sl, total, idx


def _new(src, idx, R, combine, epoch_eval='final', E=2):
    from ultrare_b200.method.sisa import Sisa
    s = Sisa(_Param(E), 'mf', len(idx), idx)
    s.epoch_eval, s.slices, s.combine, s.source = epoch_eval, R, combine, dict(src)
    return s


def _learn(src, R, combine='mean', epoch_eval='final', E=2):
    tl, sl, total, idx = _read(src, K_TOY, R)
    s = _new(src, idx, R, combine, epoch_eval, E)
    s.learn(tl, sl, total, 0, '')
    return s, (tl, sl, total)


def _snap(s):
    """Host copies of the local model state: merged table, item tables, checkpoints, combination, ledger."""
    local = [(g, m) for g, m in enumerate(s.model_list) if getattr(m, 'item_mat', None) is not None]
    c = s.combination
    return dict(P=s.model_list[0].user_mat.weight.data.cpu().numpy().copy(),
                Q={g: m.item_mat.weight.data.cpu().numpy().copy() for g, m in local},
                ck={g: [(a.cpu().numpy().copy(), b.cpu().numpy().copy()) for a, b in getattr(m, 'checkpoints', [])]
                    for g, m in local},
                comb=None if c is None else (c.w.copy(), c.b.copy(), c.T.cpu().numpy().copy(),
                                             c.b_slot.cpu().numpy().copy()),
                led=(s.deleted_users.tolist(), s.deleted_pairs.tolist()))


def _equal(a, b):
    assert np.array_equal(a['P'], b['P'])
    assert a['Q'].keys() == b['Q'].keys()
    for g in a['Q']:
        assert np.array_equal(a['Q'][g], b['Q'][g]), g
        assert len(a['ck'][g]) == len(b['ck'][g])
        for (p1, q1), (p2, q2) in zip(a['ck'][g], b['ck'][g]):
            assert np.array_equal(p1, p2) and np.array_equal(q1, q2), g
    assert (a['comb'] is None) == (b['comb'] is None)
    if a['comb'] is not None:
        for x, y in zip(a['comb'], b['comb']):
            assert np.array_equal(x, y)


def _same_metrics(a, b):
    for key in ('total_rmse', 'total_ndcg', 'total_hr'):
        assert a[key] == pytest.approx(b[key], rel=1e-12, abs=1e-12), key


def _load(d, **kw):
    from ultrare_b200.method.sisa import Sisa
    _fresh()
    return Sisa.load_state(d, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("R,combine,epoch_eval", [(1, 'mean', 'final'), (1, 'fit', 'final'), (1, 'mean', 'faithful'),
                                                  (1, 'fit', 'faithful'), (4, 'mean', 'final'), (4, 'fit', 'final')])
def test_round_trip(cuda_dev, tmp_path, R, combine, epoch_eval):
    """Learn, save, load: tables, checkpoints and the combination bit-equal; test within 1e-12; recommend bit-equal."""
    src = _toy_source(tmp_path)
    s, (tl, sl, total) = _learn(src, R, combine, epoch_eval)
    d = str(tmp_path / "s0")
    s.save_state(d)
    with pytest.raises(FileExistsError):
        s.save_state(d)
    names = sorted(os.listdir(d))
    assert 'manifest.json' in names and not any(n.endswith('.tmp') for n in names)
    assert ('ckpt0_3_P.npy' in names) == (R == 4) and ('combine.npy' in names) == (combine == 'fit')
    for n in names:
        if n.endswith('.npy'):
            np.load(os.path.join(d, n), allow_pickle=False)
    before = _snap(s)
    want = s.test(total, 0, '')
    items, scores = s.recommend(None, 10, exclude=tl)
    items, scores = items.cpu().numpy(), scores.cpu().numpy()
    L = _load(d, param=_Param(2))
    assert (L.slices, L.combine, L.epoch_eval, L.n_group) == (R, combine, epoch_eval, K_TOY)
    assert [list(g) for g in L.group_index] == [list(map(int, g)) for g in s.group_index]
    _equal(_snap(L), before)
    _same_metrics(L.test(total, 0, ''), want)
    it2, sc2 = L.recommend(None, 10, exclude=tl)
    assert np.array_equal(it2.cpu().numpy(), items) and np.array_equal(sc2.cpu().numpy(), scores)
    with pytest.raises(ValueError, match="epochs"):
        _load(d, param=_Param(3))


def _inproc_unlearn(src, before_models, idx, R, combine, users, pairs, save_dir, epoch_eval='final', prev=((), ())):
    """The in-process unlearn of a request on `before_models`: retained data = file minus prev and the request."""
    from ultrare_b200.config import routed_users
    du = list(prev[0]) + list(users)
    dp = np.concatenate([np.asarray(prev[1], dtype=np.int64).reshape(-1, 2),
                         np.asarray(pairs, dtype=np.int64).reshape(-1, 2)])
    tl, sl, total, _ = _read(src, len(idx), R, du, dp)
    s = _new(src, idx, R, combine, epoch_eval)
    s.unlearn(list(before_models), tl, sl, total, routed_users(list(users), np.asarray(pairs).reshape(-1, 2)), 0,
              save_dir)
    return s


def _pass_equal(a_dir, b_dir):
    """The artefacts of two unlearn passes: tables and slices.npy bit-equal, log0 within 1e-12."""
    names = sorted(n for n in os.listdir(a_dir) if n.startswith(('user_mat', 'item_mat', 'slices')))
    assert names == sorted(n for n in os.listdir(b_dir) if n.startswith(('user_mat', 'item_mat', 'slices')))
    for n in names:
        assert np.array_equal(np.load(os.path.join(a_dir, n)), np.load(os.path.join(b_dir, n))), n
    _same_metrics(np.load(os.path.join(a_dir, 'log0.npy'), allow_pickle=True).item(),
                  np.load(os.path.join(b_dir, 'log0.npy'), allow_pickle=True).item())
    return names


def _request(n_user=1508, seed=0, n=25):
    rs = np.random.RandomState(seed)
    return rs.choice(n_user, n, replace=False)


def _pairs(src, frac=0.02, seed=0):
    import pandas as pd
    tr = pd.read_csv(src['train_file'], header=None)
    rows = np.sort(np.random.RandomState(seed).choice(len(tr), int(frac * len(tr)), replace=False))
    return np.stack([tr[0].values[rows], tr[1].values[rows]], 1).astype(np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 4])
@pytest.mark.parametrize("kind", ["users", "pairs"])
def test_unlearn_from_a_loaded_state_equals_the_in_process_unlearn(cuda_dev, tmp_path, R, kind):
    src = _toy_source(tmp_path)
    combine = 'fit' if kind == 'pairs' else 'mean'
    s, _ = _learn(src, R, combine)
    d = str(tmp_path / "s0")
    s.save_state(d)
    users, pairs = (_request(), ()) if kind == 'users' else ((), _pairs(src))
    led = (np.unique(np.asarray(users, dtype=np.int64)).tolist(),
           np.unique(np.asarray(pairs, dtype=np.int64).reshape(-1, 2), axis=0).tolist())
    L = _load(d)
    (tmp_path / "a").mkdir()
    (tmp_path / "b").mkdir()
    eff = L.apply_request(users, pairs, save_dir=str(tmp_path / "a"))
    assert eff[0].tolist() == led[0] and eff[1].tolist() == led[1]
    _fresh()
    ref = _inproc_unlearn(src, s.model_list, s.group_index, R, combine, users, pairs, str(tmp_path / "b"))
    got, want = _snap(L), _snap(ref)
    want['led'] = led
    _equal(got, want)
    assert got['led'] == want['led'] and L.requests == 1
    assert L.log['train_loss'] == ref.log['train_loss']
    assert L.retrain_gid == ref.retrain_gid and len(L.retrain_gid) > 0
    if R > 1:
        assert L.first_slice.tolist() == ref.first_slice.tolist()
    _same_metrics(L.final_log, ref.final_log)
    _pass_equal(str(tmp_path / "a"), str(tmp_path / "b"))


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 4])
def test_two_requests_across_a_save_and_load(cuda_dev, tmp_path, R):
    """A, save, load, B equals the in-process A then B; for R = 4 it agrees with a sliced learn on the data minus
    A and B; repeating A retrains nothing and leaves the state bit-equal."""
    src = _toy_source(tmp_path)
    s, _ = _learn(src, R, 'fit')
    s.save_state(str(tmp_path / "s0"))
    A = np.sort(_request(seed=1, n=20))
    every = _pairs(src, 1.0)
    B_pairs = np.concatenate([_pairs(src, 0.01, seed=2), every[np.isin(every[:, 0], A)][:5]])    # 5 pairs of A's users
    L = _load(str(tmp_path / "s0"))
    L.apply_request(A, ())
    L.save_state(str(tmp_path / "s1"))
    L = _load(str(tmp_path / "s1"))
    assert L.requests == 1 and L.deleted_users.tolist() == A.tolist()
    eu, ep = L.apply_request((), B_pairs)
    assert len(eu) == 0 and not np.isin(ep[:, 0], A).any()        # the pairs of A's users were dropped
    L.save_state(str(tmp_path / "s2"))
    _fresh()
    r1 = _inproc_unlearn(src, s.model_list, s.group_index, R, 'fit', A, (), '')
    r2 = _inproc_unlearn(src, r1.model_list, s.group_index, R, 'fit', (), ep, '', prev=(A, ()))
    got, want = _snap(L), _snap(r2)
    want['led'] = got['led']
    _equal(got, want)
    _same_metrics(L.final_log, r2.final_log)
    assert L.deleted_users.tolist() == A.tolist()
    assert L.deleted_pairs.tolist() == np.unique(ep, axis=0).tolist() and L.requests == 2
    if R == 4:
        tl, sl, total, idx = _read(src, K_TOY, R, A, ep)
        ref = _new(src, idx, R, 'fit')
        ref.learn(tl, sl, total, 0, '')
        b = _snap(ref)
        assert np.abs(got['P'] - b['P']).max() < 1e-4
        for g in got['Q']:
            assert np.abs(got['Q'][g] - b['Q'][g]).max() < 1e-4
        assert L.final_log['total_rmse'] == pytest.approx(ref.final_log['total_rmse'], rel=1e-3)
    # a repeated request: nothing retrained, the saved state bit-equal
    L = _load(str(tmp_path / "s2"))
    eu, ep2 = L.apply_request(A[:3], ep[:2])
    assert len(eu) == 0 and len(ep2) == 0 and L.retrain_gid == set()
    L.save_state(str(tmp_path / "s3"))
    for n in sorted(os.listdir(tmp_path / "s2")):
        a, b = tmp_path / "s2" / n, tmp_path / "s3" / n
        assert a.read_bytes() == b.read_bytes(), n


class _Ranks:
    """Ranks as threads on one GPU (test_combine._ThreadDist, plus the barrier save_state needs); the device copies
    of each call are made one thread at a time, as the training launches are."""

    def __init__(self, world):
        from test_combine import _ThreadDist

        class Dist(_ThreadDist):
            def barrier(self):
                self.sh["barrier"].wait()
        self.world, self.Dist = world, Dist
        self.shared = dict(barrier=threading.Barrier(world), slots=[None] * world)
        self.lock = threading.RLock()

    def dist(self, r):
        return self.Dist(r, self.world, self.shared)

    def run(self, fn):
        out, errs = [None] * self.world, []

        def one(r):
            try:
                out[r] = fn(r)
            except BaseException as e:          # noqa: BLE001 -- re-raised below; the other ranks are released
                errs.append(e)
                self.shared["barrier"].abort()
        th = [threading.Thread(target=one, args=(r,)) for r in range(self.world)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errs:
            raise errs[0]
        return out

    def serialise(self, monkeypatch, sisa):
        from ultrare_b200 import kernels as kn
        lock = self.lock
        for name in ('download_many', 'upload_table'):
            f = getattr(kn, name)

            def locked(*a, _f=f, **k):
                with lock:
                    return _f(*a, **k)
            monkeypatch.setattr(kn, name, locked)
        for name in ('_train_sliced', '_train_shards'):
            f = getattr(type(sisa), name)

            def locked_m(self, *a, _f=f, **k):
                with lock:
                    return _f(self, *a, **k)
            monkeypatch.setattr(type(sisa), name, locked_m)


@pytest.mark.gpu
def test_world_size_save_at_two_load_at_one_and_three(cuda_dev, tmp_path, monkeypatch):
    """A state saved by 2 ranks loads at 1 and at 3 ranks; the unlearn from it equals the in-process unlearn at that
    world size and agrees with one GPU within the training tolerances."""
    from ultrare_b200.method.sisa import Sisa, _RemoteModel
    src = _toy_source(tmp_path)
    R, combine = 4, 'fit'
    s, _ = _learn(src, R, combine)
    keep_P = s.model_list[0].user_mat.weight
    du = np.sort(np.random.RandomState(0).choice(1508, 30, replace=False))
    tl, sl, total, _ = _read(src, K_TOY, R, du)
    ranks2 = _Ranks(2)
    ranks2.serialise(monkeypatch, s)
    d = str(tmp_path / "s2ranks")

    def save(r):
        sr = Sisa.__new__(Sisa)
        sr.__dict__.update(s.__dict__)
        sr._writers = []
        sr.dist = ranks2.dist(r)
        sr.model_list = [m if k % 2 == r else _RemoteModel(keep_P) for k, m in enumerate(s.model_list)]
        sr.save_state(d)
    ranks2.run(save)
    assert json.load(open(os.path.join(d, 'manifest.json')))['saved_world_size'] == 2
    # one GPU: loaded vs in-process
    L1 = _load(d)
    L1.apply_request(du, (), tl, sl, total)
    one = _snap(L1)
    ref1 = _inproc_unlearn(src, s.model_list, s.group_index, R, combine, du, (), '')
    want = _snap(ref1)
    want['led'] = one['led']
    _equal(one, want)
    _same_metrics(L1.final_log, ref1.final_log)
    # three ranks: loaded vs in-process
    for m in s.model_list:
        m.user_mat.weight = keep_P
    _fresh()
    ranks3 = _Ranks(3)
    ranks3.lock = ranks2.lock

    def loaded(r):
        from ultrare_b200.method.sisa import Sisa as S
        L = S.load_state(d, dist=ranks3.dist(r))
        L.apply_request(du, (), tl, sl, total)
        return _snap(L), dict(L.final_log)
    got = ranks3.run(loaded)
    ranks3b = _Ranks(3)
    ranks3b.lock = ranks2.lock

    def inproc(r):
        sr = _new(src, s.group_index, R, combine)
        sr.dist = ranks3b.dist(r)
        models = [m if k % 3 == r else _RemoteModel(keep_P) for k, m in enumerate(s.model_list)]
        sr.unlearn(models, tl, sl, total, du.tolist(), 0, '')
        return _snap(sr), dict(sr.final_log)
    want3 = ranks3b.run(inproc)
    for r in range(3):
        (g, glog), (w, wlog) = got[r], want3[r]
        w['led'] = g['led']
        _equal(g, w)
        _same_metrics(glog, wlog)
        assert np.abs(g['P'] - one['P']).max() < 1e-4, r
        for k, q in g['Q'].items():
            assert np.abs(q - one['Q'][k]).max() < 1e-4, (r, k)
        assert glog['total_rmse'] == pytest.approx(L1.final_log['total_rmse'], rel=1e-3)


# ------------------------------------------------------------------------------------------------------------ CLI
def _main(env, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "main.py"), *args], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("deltype", ["rand", "inter"])
def test_cli_request_runs_end_to_end(cuda_dev, tmp_path, deltype):
    """--save-state on the group run, then the scripted deletion set as a request run from the learn pass's state in a
    separate process: the same retrained tables and slices.npy as the scripted unlearn pass, log0 within 1e-12; then
    a second request from the request run's state, whose ledger holds both."""
    env = dict(os.environ, ULTRARE_ROOT=str(tmp_path))
    _main(env, "--dataset", "ml1m", "--synth", "--group", "5", "--slices", "4", "--grouping", "rating-ot", "--epoch",
          "2", "--verbose", "0", "--deltype", deltype, "--save-state", "--recommend", "5")
    gdir = tmp_path / "result" / "2" / deltype / "ml1m_g5"
    learn, unlearn = gdir / "MF_rating-ot_sisa_learn", gdir / "MF_rating-ot_sisa_unlearn"
    dele = np.load(gdir / "deletion.npy", allow_pickle=True)
    del_user, del_rating = np.asarray(dele[0], dtype=np.int64), np.asarray(dele[1], dtype=np.int64).reshape(-1, 2)
    assert (len(del_user) > 0) == (deltype == "rand") and (len(del_rating) > 0) == (deltype == "inter")
    for sub in (learn, unlearn):
        assert (sub / "state" / "manifest.json").exists()
    man = json.loads((learn / "state" / "manifest.json").read_text())
    assert (man['K'], man['slices'], man['dataset'], man['grouping'], man['requests']) == (5, 4, 'ml1m', 'rating-ot', 0)
    led = np.load(unlearn / "state" / "deleted_users.npy"), np.load(unlearn / "state" / "deleted_pairs.npy")
    assert led[0].tolist() == np.unique(del_user).tolist() and \
        led[1].tolist() == np.unique(del_rating.reshape(-1, 2), axis=0).tolist()
    out = tmp_path / "req1"
    if deltype == "rand":
        f = tmp_path / "users.txt"
        f.write_text("\n".join(str(int(u)) for u in del_user) + "\n")
        req = ["--forget-users", str(f)]
    else:
        f = tmp_path / "ratings.csv"
        f.write_text("".join(f"{int(u)},{int(i)}\n" for u, i in del_rating))
        req = ["--forget-ratings", str(f)]
    _main(env, "--unlearn-from", str(learn / "state"), "--out", str(out), "--verbose", "0", "--recommend", "5", *req)
    names = _pass_equal(str(out), str(unlearn))
    assert "slices.npy" in names and any(n.startswith("item_mat") for n in names)
    assert np.array_equal(np.load(out / "rec5.npy"), np.load(unlearn / "rec5.npy"))
    eff = np.load(out / "deletion.npy", allow_pickle=False)
    assert eff.dtype == np.int64 and eff.shape[1] == 2
    for n in os.listdir(unlearn / "state"):                  # the request's state is the scripted pass's state
        if n.endswith('.npy'):
            assert np.array_equal(np.load(out / "state" / n), np.load(unlearn / "state" / n)), n
    assert (learn / "state" / "manifest.json").read_text() == json.dumps(man, indent=1)   # the input state untouched
    # a second request from the first request's state
    second = np.setdiff1d(np.arange(0, 6040, 97), del_user)[:12]
    np.save(tmp_path / "second.npy", second)
    _main(env, "--unlearn-from", str(out / "state"), "--out", str(tmp_path / "req2"), "--verbose", "0",
          "--forget-users", str(tmp_path / "second.npy"))
    st2 = tmp_path / "req2" / "state"
    assert np.load(st2 / "deleted_users.npy").tolist() == np.union1d(del_user, second).tolist()
    assert np.load(st2 / "deleted_pairs.npy").tolist() == led[1].tolist()
    assert json.loads((st2 / "manifest.json").read_text())['requests'] == 2
    # the same request again: nothing to do, the state carries over unchanged
    stdout = _main(env, "--unlearn-from", str(st2), "--out", str(tmp_path / "req3"), "--verbose", "0",
                   "--forget-users", str(tmp_path / "second.npy"))
    assert "no shard is retrained" in stdout
    for n in os.listdir(st2):
        assert (st2 / n).read_bytes() == (tmp_path / "req3" / "state" / n).read_bytes(), n
