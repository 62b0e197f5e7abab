"""CPU: the host-only half of the native batch runtime (csrc/mf_batch.cu, the host entry points of
csrc/mf_train_owner.cu) -- layout of a K-shard batch inside one allocation, apportioning of the training CTAs to the
shards, plan -> launch parameters.  None of these calls touches the device (pointer arithmetic on the arena base
only), so they run without a GPU; the kernels that consume the layout are the -m gpu tests' business."""
import ctypes as C

import numpy as np
import pytest

ML1M_SHARDS = [(181_204, 1208), (176_377, 1208), (179_981, 1208), (174_210, 1208), (163_000, 1208)]   # (n, n_user)


def _lib():
    from ultrare_b200 import _lib
    return _lib, _lib.lib()


def _shards(L, spec, perm=None):
    hs = (L.MFBatchShard * len(spec))()
    for j, (n, nu) in enumerate(spec):
        hs[j].inter, hs[j].perm = 0x10000000 + 0x1000000 * j, (perm if perm else None)
        hs[j].n, hs[j].n_user, hs[j].shard_id, hs[j].group = n, nu, j + 1, j & 1
    return hs


def _layout(spec, n_item=3416, d=16, batch=30_000, epochs=50, owner=1, sched_cap=512 << 20, perm=None):
    L, h = _lib()
    lay = L.MFBatchLayout()
    rc = h.ure_mf_batch_layout(_shards(L, spec, perm), len(spec), n_item, d, batch, epochs, owner, sched_cap, C.byref(lay))
    return rc, lay


def test_batch_layout_regions_are_aligned_disjoint_and_large_enough():
    L, h = _lib()
    K, I, d, B, E = len(ML1M_SHARDS), 3416, 16, 30_000, 50
    rc, lay = _layout(ML1M_SHARDS, I, d, B, E)
    assert rc == 0 and lay.owner == 1 and lay.grid >= 1
    rows = sum(nu for _, nu in ML1M_SHARDS)
    n_tot = sum(n for n, _ in ML1M_SHARDS)
    table_rows = rows + K * I
    assert (lay.rows_total, lay.n_total) == (rows, n_tot)
    assert lay.spe_cap == max(-(-n // B) for n, _ in ML1M_SHARDS) == 7
    assert lay.max_rows == max(I, max(nu for _, nu in ML1M_SHARDS)) and lay.max_n == max(n for n, _ in ML1M_SHARDS)
    assert lay.sched_stride == 2 * n_tot and 2 <= lay.sched_rows <= E + 1
    # every region starts on a 256-byte boundary, in this order, and holds what its consumer indexes
    order = ["table", "W", "ws", "Z", "sse", "off", "zero_end", "rec", "radix", "perm_inv", "sched", "sched_off", "total"]
    offs = [getattr(lay, nm) for nm in order]
    assert all(o % 256 == 0 for o in offs) and offs == sorted(offs) and offs[0] == 0
    size = {a: getattr(lay, b) - getattr(lay, a) for a, b in zip(order, order[1:])}
    assert size["table"] >= K * C.sizeof(L.MFShard)
    assert size["W"] >= table_rows * d * 4 and size["Z"] >= 2 * table_rows * d * 4
    assert size["ws"] >= h.ure_mf_train_workspace_bytes()
    assert size["sse"] >= K * E * 8
    assert size["off"] >= sum(nu + I + 4 for _, nu in ML1M_SHARDS) * 4
    assert size["rec"] >= 4 * n_tot * 16                          # user-sorted, item-sorted, two radix scratch copies
    assert size["radix"] >= h.ure_mf_owner_radix_bytes(K)
    assert size["perm_inv"] == 0                                  # no explicit visiting orders
    assert size["sched"] >= lay.sched_rows * lay.sched_stride * 2
    assert size["sched_off"] >= lay.sched_rows * lay.grid * (lay.spe_cap + 1) * 4
    # explicit visiting orders: room for their inverses, one int per record and epoch
    rc, lay_p = _layout(ML1M_SHARDS, I, d, B, E, perm=0x7000000)
    assert rc == 0 and lay_p.sched - lay_p.perm_inv >= E * n_tot * 4


def test_batch_layout_schedule_window_follows_the_memory_cap():
    """The schedule tables take at most `sched_bytes_cap`: fewer resident epochs (>= 2 rows), never more than
    epochs + 1 rows."""
    rc, big = _layout(ML1M_SHARDS, epochs=50)
    rc2, small = _layout(ML1M_SHARDS, epochs=50, sched_cap=1)
    rc3, few = _layout(ML1M_SHARDS, epochs=3)
    assert rc == rc2 == rc3 == 0
    assert big.sched_rows == 51 and small.sched_rows == 2 and few.sched_rows == 4
    assert small.total < big.total


def test_batch_layout_refuses_the_owner_schedule_when_row_state_exceeds_shared_memory():
    # C4-shaped: 8 shards x (1.25 M users + 1 M items) x d = 128 -- far beyond 148 x 200 KB
    rc, lay = _layout([(15_000_000, 1_250_000)] * 8, n_item=1_000_000, d=128)
    assert rc == 0 and lay.owner == 0 and lay.rec == 0 and lay.sched == 0 and lay.total == lay.zero_end
    rc, lay = _layout(ML1M_SHARDS, owner=0)                       # not asked for
    assert rc == 0 and lay.owner == 0
    rc, lay = _layout([(0, 10), (0, 12)])                         # nothing to train
    assert rc == 0 and lay.owner == 0


def test_batch_layout_rejects_bad_arguments_with_a_message():
    L, h = _lib()
    lay = L.MFBatchLayout()
    for spec, n_item, d, batch in (([(-1, 5)], 10, 16, 100), ([(5, 0)], 10, 16, 100), ([(5, 5)], 0, 16, 100),
                                   ([(5, 5)], 10, 0, 100), ([(5, 5)], 10, 16, 0)):
        rc = h.ure_mf_batch_layout(_shards(L, spec), len(spec), n_item, d, batch, 2, 1, 1 << 20, C.byref(lay))
        assert rc != 0 and b"ure_mf_batch_layout" in h.ure_last_error()
    too_many = L.URE_MAX_SHARDS + 1
    rc = h.ure_mf_batch_layout(_shards(L, [(5, 5)] * too_many), too_many, 10, 16, 100, 2, 1, 1 << 20, C.byref(lay))
    assert rc != 0                                                # more than URE_MAX_SHARDS
    rc, lay = _layout([(50, 5)] * L.URE_MAX_SHARDS)               # more shards than SMs: no owner schedule (one CTA each at least)
    assert rc == 0 and (lay.owner == 0 or lay.grid >= L.URE_MAX_SHARDS)


def _plan(lay, plan, d=16, allow_cache=1, force=(-1, 0)):
    L, h = _lib()
    hp = L.MFHParams(d=d, batch=30_000, lr0=1e-3, lr_decay=0.95, lr_step=50, weight_decay=0.1, momentum=0.9, mode=L.MF_DENSE)
    info = (C.c_int32 * 8)()
    arr = (C.c_int32 * 4)(*plan)
    base = 1 << 32
    rc = h.ure_mf_batch_plan(arr, 5, C.byref(hp), C.c_void_p(base), C.byref(lay), allow_cache, force[0], force[1], info)
    return rc, hp, list(info), base


def test_batch_plan_picks_the_fastest_shared_memory_configuration_that_fits():
    L, h = _lib()
    _, lay = _layout(ML1M_SHARDS)
    avail = 227 << 10
    # ml1m-sized plan: 120 owned rows, ~12 k owned slots per CTA, 7 steps per epoch -> the record cache fits
    rc, hp, info, base = _plan(lay, (120, 11_990, 7, avail))
    assert rc == 1 and hp.mode == L.MF_OWNER
    assert (hp.owner_cap_rows, hp.owner_cap_slots, hp.owner_flags, hp.owner_cap_list) == (120, 12_000, 1, 12_000)
    assert hp.owner_spe_cap == lay.spe_cap and hp.owner_sched_rows == lay.sched_rows and hp.owner_sched_stride == lay.sched_stride
    assert hp.owner_sched == base + lay.sched and hp.owner_sched_off == base + lay.sched_off and hp.owner_max_n == lay.max_n
    need = h.ure_mf_owner_smem_bytes(16, 120, 12_000, 12_000, 7, 1)
    assert info[:6] == [1, 1, 12_000, 120, 12_000, 7] and info[6] == need <= avail == info[7]
    # the cache forbidden, or too little shared memory for it: staged lists, as many entries as fit (multiple of 16)
    rc, hp, info, _ = _plan(lay, (120, 11_990, 7, avail), allow_cache=0)
    assert rc == 1 and hp.owner_flags == 0 and hp.owner_cap_list == 12_000
    tight = int(h.ure_mf_owner_smem_bytes(16, 120, 12_000, 16, 7, 0)) + 160 * 100
    rc, hp, info, _ = _plan(lay, (120, 11_990, 7, tight))
    assert rc == 1 and hp.owner_flags == 0 and 1024 <= hp.owner_cap_list < 12_000 and hp.owner_cap_list % 16 == 0
    assert h.ure_mf_owner_smem_bytes(16, 120, 12_000, hp.owner_cap_list, 7, 0) <= tight
    # not even sixteen staged entries fit: the plan is refused and the launch parameters stay untouched
    rc, hp, info, _ = _plan(lay, (120, 11_990, 7, 4096))
    assert rc == 0 and info[0] == 0 and hp.mode == L.MF_DENSE and hp.owner_sched is None
    # capacities the kernels cannot index: 16-bit slot numbers, 12-bit row numbers
    assert _plan(lay, (120, 70_000, 7, 1 << 30))[0] == 0
    assert _plan(lay, (5000, 11_990, 7, 1 << 30))[0] == 0
    # a forced configuration (test hook) is honoured when it fits
    rc, hp, info, _ = _plan(lay, (120, 11_990, 7, avail), force=(2, 2048))
    assert rc == 1 and hp.owner_flags == 2 and hp.owner_cap_list == 2048


def test_owner_smem_bytes_grows_with_every_capacity():
    _, h = _lib()
    base = h.ure_mf_owner_smem_bytes(16, 100, 8000, 8000, 7, 1)
    assert base > 0
    assert h.ure_mf_owner_smem_bytes(16, 101, 8000, 8000, 7, 1) > base
    assert h.ure_mf_owner_smem_bytes(16, 100, 8016, 8016, 7, 1) > base
    assert h.ure_mf_owner_smem_bytes(64, 100, 8000, 8000, 7, 1) > base
    assert h.ure_mf_owner_smem_bytes(16, 100, 8000, 4000, 7, 0) < h.ure_mf_owner_smem_bytes(16, 100, 8000, 8000, 7, 0)


def test_host_stage_copy_copies_every_size_and_requires_an_aligned_destination():
    """ure_host_stage_copy (non-temporal stores into page-locked staging memory; the host half of every upload): 64-byte
    main loop, 16-byte loop, byte tail; any source alignment; a destination off the 16-byte grid is an error."""
    _, h = _lib()
    rng = np.random.default_rng(1)
    src_all = rng.integers(0, 256, 1_000_200, dtype=np.uint8)
    raw = np.zeros(1_000_200 + 64, dtype=np.uint8)
    o = (-raw.ctypes.data) % 64
    dst_all = raw[o:o + 1_000_200]
    assert dst_all.ctypes.data % 64 == 0
    for nbytes in (0, 1, 15, 16, 17, 63, 64, 65, 4097, 1_000_003):
        for soff in (0, 1, 7, 16):
            dst_all[:] = 0
            src = src_all[soff:soff + nbytes]
            assert h.ure_host_stage_copy(C.c_void_p(dst_all.ctypes.data), C.c_void_p(src.ctypes.data), nbytes) == 0
            assert np.array_equal(dst_all[:nbytes], src) and not dst_all[nbytes:nbytes + 64].any()
    assert h.ure_host_stage_copy(C.c_void_p(dst_all.ctypes.data + 8), C.c_void_p(src_all.ctypes.data), 64) != 0
    assert b"16-byte aligned" in h.ure_last_error()


def test_scratch_size_queries_are_positive_and_monotone():
    """The *_bytes entry points a caller sizes its scratch tensors with (host-only)."""
    _, h = _lib()
    assert h.ure_mf_train_workspace_bytes() > 0 and h.ure_sinkhorn_workspace_bytes() > 0
    assert 0 < h.ure_mf_owner_radix_bytes(1) < h.ure_mf_owner_radix_bytes(5)
    assert h.ure_partition_blocks() >= 1
