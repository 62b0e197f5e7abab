"""CPU: the C-ABI library builds for sm_100a, loads, and exports every symbol include/ultrare_b200.h declares
(no compute calls: there is no GPU here); the product never imports the oracle."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_are_exported_and_bound():
    from ultrare_b200 import _lib, build
    path = build.build()
    header = open(os.path.join(ROOT, "include", "ultrare_b200.h")).read()
    declared = set(re.findall(r"\b(ure_[a-z0-9_]+)\s*\(", header))
    handle = ctypes.CDLL(path)
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in the header but not exported"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert handle.ure_abi_version() == 7
    handle.ure_last_error.restype = ctypes.c_char_p
    assert isinstance(handle.ure_last_error(), bytes)


def test_struct_layouts_match_the_header():
    from ultrare_b200 import _lib
    assert ctypes.sizeof(_lib.MFShard) == 176 and ctypes.sizeof(_lib.MFHParams) == 136
    assert _lib.MFShard.inter_u.offset == 96 and _lib.MFShard.n.offset == 152 and _lib.MFShard.perm_seed.offset == 168
    assert _lib.MFHParams.mode.offset == 28 and _lib.MFHParams.decay.offset == 32 and _lib.MFHParams.owner_cap_rows.offset == 44


def test_sass_has_blackwell_tensor_and_bulk_copy_instructions():
    """tcgen05.mma -> UTC*MMA, tcgen05.ld -> LDTM, cp.async.bulk -> UBLKCP, red.v4.f32 -> REDG...F32x4."""
    from ultrare_b200 import build
    so = os.path.join(ROOT, "ultrare_b200", "libultrare_b200.so")
    cuobjdump = os.path.join(os.path.dirname(build.NVCC), "cuobjdump")      # the toolkit that built the library
    sass = subprocess.run([cuobjdump, "-sass", so], capture_output=True, text=True).stdout
    assert re.search(r"UTC[A-Z]*MMA", sass), "no tcgen05 MMA in SASS"
    assert "LDTM" in sass and "UBLKCP" in sass
    assert re.search(r"RED[G]?\.E\.ADD\.F32x4", sass)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "ultrare_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), os.path.join(dp, f)


def test_cuda_required_loudly():
    import torch
    if torch.cuda.is_available():
        return
    import pytest
    from ultrare_b200.method.utils import MF
    from ultrare_b200 import kernels as kn
    with pytest.raises(RuntimeError):
        MF(10, 10, 16)
    with pytest.raises(RuntimeError):
        kn.ensemble_score([torch.zeros(4, 16)], [torch.zeros(4, 16)], torch.zeros((1, 4), dtype=torch.int32))


def test_host_read_rating_matches_oracle():
    """ultrare_b200.read.readRating (owner-map single pass) == oracle restatement of read.py:9-70."""
    import numpy as np
    import pandas as pd
    from oracle import sisa as osisa
    from ultrare_b200.read import readRating
    rng = np.random.default_rng(0)
    n_user, n = 200, 5000
    u = np.sort(rng.integers(0, n_user, n))
    i = rng.integers(0, 300, n)
    r = rng.integers(1, 6, n).astype(float)
    groups = osisa.uniform_groups(n_user, 4)
    dels = rng.choice(n_user, 15, replace=False)
    for sort in ("a", "r"):
        got, gidx = readRating(pd.DataFrame({0: u, 1: i, 2: r}), n_user, 5, list(dels), [], 4, groups, sort)
        ref, ridx = osisa.read_rating(u, i, r, n_user, 5, dels, 4, groups, sort)
        assert [list(a) for a in gidx] == [list(a) for a in ridx]
        for a, b in zip(got, ref):
            assert a.shape == b.shape and np.array_equal(a, b)


def test_device_rating_data_host_views_match_host_read_rating():
    """The host-side views of a device-backed RatingData (users / items / ratings / _raw, rebuilt on demand from the
    source table without touching the device) equal what readRating returns for the same groups and deletions."""
    import pandas as pd
    import torch
    from ultrare_b200.read import DeviceRatingData, readRating
    rng = np.random.default_rng(9)
    n_user, n = 90, 4000
    df = pd.DataFrame({0: rng.integers(0, n_user, n), 1: rng.integers(0, 40, n), 2: rng.integers(1, 6, n)})
    del_user = [3, 17, 42]
    host, groups = readRating(df, n_user, 5, del_user, [], 4, [], 'a')
    owner = np.full(n_user, -1, dtype=np.int32)
    for g in range(3, -1, -1):
        owner[np.asarray(groups[g])] = g
    deleted = np.zeros(n_user, dtype=np.uint8)
    deleted[del_user] = 1
    src = (df, owner, deleted, 5.0)
    for g in range(4):
        ds = DeviceRatingData(torch.zeros((host[g].shape[1], 4), dtype=torch.int32), src, (g, g + 1))
        assert len(ds) == host[g].shape[1]
        assert np.array_equal(ds._raw, host[g])
        assert np.array_equal(ds.users, host[g][0].astype(int)) and np.array_equal(ds.items, host[g][1].astype(int))
        assert np.array_equal(ds.ratings, host[g][2])
    total = DeviceRatingData(torch.zeros((sum(h.shape[1] for h in host), 4), dtype=torch.int32), src, (0, 4))
    assert np.array_equal(total._raw, np.hstack(host))


def test_pack_threads_follow_ranks_per_node(monkeypatch):
    from ultrare_b200 import kernels as kn
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 8)
    monkeypatch.delenv("URE_PACK_THREADS", raising=False)
    monkeypatch.setenv("LOCAL_WORLD_SIZE", "1")
    assert kn._default_pack_threads() == max(1, min(8, cores - 1))
    monkeypatch.setenv("LOCAL_WORLD_SIZE", str(cores))
    assert kn._default_pack_threads() == 1
    monkeypatch.setenv("URE_PACK_THREADS", "5")
    assert kn._default_pack_threads() == 5


def test_cli_keeps_the_reference_flags_defaults_and_checks():
    """main.py's argparse surface (reference main.py:5-14): same flags, same defaults, AssertionError on the values
    the reference's asserts reject (main.py:21-53)."""
    import pytest
    from ultrare_b200.main import _checked, parser
    d = vars(parser.parse_args([]))
    assert {k: d[k] for k in ('dataset', 'epoch', 'worker', 'verbose', 'group', 'layer', 'learn', 'delper', 'deltype')} == \
        dict(dataset='ml1m', epoch=50, worker=24, verbose=1, group=2, layer=[64, 32], learn='sisa', delper=2,
             deltype='rand')
    ok = _checked(parser.parse_args('--dataset ml1m --epoch 50 --group 5 --learn sisa --delper 5 --deltype rand'.split()))
    assert ok.group == 5 and ok.delper == 5
    for bad in ('--delper 3', '--epoch 0', '--verbose 7', '--learn seq', '--deltype core', '--group -1', '--dataset ml20m'):
        with pytest.raises(AssertionError):
            _checked(parser.parse_args(bad.split()))


def test_instance_read_data_host_branch(tmp_path, monkeypatch):
    """Instance._read_data without a CUDA device (or with URE_HOST_INGEST=1) is the host split of `_read`
    (config.py:80-96): RatingData per group, the merged test set = their concatenation."""
    import ultrare_b200.config as cfg
    import ultrare_b200.group as grp
    from ultrare_b200 import synth
    data, save = str(tmp_path / "data"), str(tmp_path / "result")
    for mod in (cfg, grp):
        monkeypatch.setattr(mod, "DATA_DIR", data)
        monkeypatch.setattr(mod, "SAVE_DIR", save)
    monkeypatch.setenv("URE_HOST_INGEST", "1")
    synth.ensure_dataset("toy")
    ins = cfg.Instance(cfg.InsParam("toy", 2, 1, [32], 3, 2, "rand"))
    train, idx, test, total = ins._read_data(True, 3, [])
    raw_train, raw_idx, raw_test = ins._read(True, 3, [])
    assert [list(g) for g in idx] == [list(g) for g in raw_idx] and len(train) == len(test) == 3
    for g in range(3):
        assert np.array_equal(train[g]._raw, raw_train[g]) and np.array_equal(test[g]._raw, raw_test[g])
    assert len(total) == sum(len(t) for t in test) and np.array_equal(total._raw, np.hstack(raw_test))
    deleted = set(int(u) for u in ins.param.del_user)
    assert not deleted & set(int(u) for t in train for u in np.unique(t.users))


def test_upload_ring_host_logic(monkeypatch):
    """kernels._upload_ring (uploads beyond UPLOAD_ONE_SHOT_BYTES): segment hand-over, ragged tail, both segments back
    in the staging pool -- with the real ure_host_stage_copy, the DMA stood in by memmove and events by no-ops (the
    GPU version of this test is test_uploads_through_the_staging_ring_equal_one_shot_uploads)."""
    import torch
    from ultrare_b200 import _lib, kernels as kn
    real = _lib.lib()
    waits = []

    class Lib:
        def __getattr__(self, name):
            return getattr(real, name)

        def ure_copy_to_device_async(self, dst, src, n, stream):
            ctypes.memmove(dst, src, n)
            return 0

    class Event:
        def record(self, *a):
            pass

        def synchronize(self):
            waits.append(1)

        def query(self):
            return True

    fake = Lib()
    monkeypatch.setattr(kn._lib, "lib", lambda: fake)
    monkeypatch.setattr(torch.cuda, "Event", Event)
    monkeypatch.setattr(kn, "_stream", lambda: None)
    monkeypatch.setattr(kn, "_staging_bytes", lambda nb: torch.empty(1 << max(12, int(nb - 1).bit_length()), dtype=torch.uint8))
    monkeypatch.setattr(kn, "_PINNED_BYTES", {})
    monkeypatch.setattr(kn, "UPLOAD_RING_BYTES", (1 << 22) + (1 << 20))
    rng = np.random.default_rng(0)
    for count in (3 * (1 << 20) + 12345, 1000, 655360 + 1):       # 5 segments and a tail; one short segment; one + 8 bytes
        src = rng.standard_normal(count)
        dst = np.zeros_like(src)
        waits.clear()
        kn._upload_ring(dst.ctypes.data, src.ctypes.data, src.nbytes)
        assert np.array_equal(src, dst)
        n_seg = -(-src.nbytes // kn.UPLOAD_RING_BYTES)
        assert len(waits) == max(0, n_seg - 2)                      # a segment is waited for only before its re-use
    assert sum(len(v) for v in kn._PINNED_BYTES.values()) == 6      # two segments returned per upload


def test_staging_pools_take_a_free_buffer_behind_a_busy_one(monkeypatch):
    """The page-locked staging pools hand out the first buffer whose last copy has completed.  With uploads on two
    streams the FIRST entry can still be busy when a later one is free; taking that one out with list.remove compared
    (tensor, event) tuples element-wise and raised "Boolean value of Tensor ... is ambiguous" (2-GPU run of the round)."""
    import torch
    from ultrare_b200 import kernels as kn

    class Event:
        def __init__(self, done):
            self.done = done

        def query(self):
            return self.done

    a, b, c = (torch.full((4096,), v, dtype=torch.uint8) for v in (0, 1, 2))
    pool = [(a, Event(False)), (b, Event(True)), (c, None)]
    monkeypatch.setattr(kn, "_PINNED_BYTES", {4096: pool})
    assert kn._staging_bytes(16) is b and [x[0] is y for x, y in zip(pool, (a, c))] == [True, True]
    assert kn._staging_bytes(4096) is c and len(pool) == 1 and pool[0][0] is a
    ra, rb = torch.zeros((1024, 4), dtype=torch.int32), torch.ones((1024, 4), dtype=torch.int32)
    rpool = [(ra, Event(False)), (rb, Event(True))]
    monkeypatch.setattr(kn, "_PINNED", {1024: rpool})
    assert kn._staging(1000) is rb and len(rpool) == 1 and rpool[0][0] is ra
