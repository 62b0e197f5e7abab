"""Tensor-level wrappers over the C ABI (include/ultrare_b200.h).

PyTorch is used for device memory and streams only; every arithmetic step on the
hot path is a hand-written sm_100a kernel inside libultrare_b200.so.  All calls are
asynchronous on the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import time
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import MFHParams, MFShard, check


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


_SIDE_STREAMS = {}


def side_stream(device, lane: int = 0) -> "torch.cuda.Stream":
    """Extra streams per device for copies that must not queue behind a long kernel on the caller's stream: lane 0
    carries uploads, lane 1 the read-backs that wait for that kernel (so that uploads never queue behind them)."""
    dev = torch.device(device)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    if (idx, lane) not in _SIDE_STREAMS:
        _SIDE_STREAMS[(idx, lane)] = torch.cuda.Stream(device=idx)
    return _SIDE_STREAMS[(idx, lane)]


SIDE_SMALL_UPLOADS = True      # pointer tables / flags of the merge and the evaluation travel on the side stream


def on_side(device):
    """Context: torch work inside runs on the upload side stream; on exit the caller's stream waits for it.  Tensors
    allocated inside must be handed to the caller's stream with record_stream (see upload_array)."""
    import contextlib

    @contextlib.contextmanager
    def ctx():
        main = torch.cuda.current_stream(device)
        side = side_stream(device)
        with torch.cuda.stream(side):
            yield main
        main.wait_stream(side)
    return ctx()


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("ultrare_b200: tensors must live on a CUDA device (no CPU path exists)")


# ------------------------------------------------------------------------------ interactions
def _default_pack_threads() -> int:
    """Staging-copy threads of this process: 8, or this rank's share of the host cores when several ranks run on
    the node (8 ranks x 8 copy threads on a 16-core host made the end-to-end step 3x slower)."""
    import os
    if "URE_PACK_THREADS" in os.environ:
        return max(1, int(os.environ["URE_PACK_THREADS"]))
    local = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1"))))
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 8)
    return max(1, min(8, cores // local - 1))


_PACK_THREADS = _default_pack_threads()
_POOL = []


def _pack_pool():
    if not _POOL:
        from concurrent.futures import ThreadPoolExecutor
        _POOL.append(ThreadPoolExecutor(max_workers=_PACK_THREADS))
    return _POOL[0]


_PINNED = {}   # rows -> list of pinned int32 [rows,4] staging buffers (reused: cudaHostAlloc is slow)


def _staging(n: int) -> torch.Tensor:
    cap = 1 << max(10, int(n - 1).bit_length())
    pool = _PINNED.setdefault(cap, [])
    for idx, (buf, ev) in enumerate(pool):
        if ev is None or ev.query():
            del pool[idx]                # by position: list.remove would compare the tensors of the entries before it
            return buf
    return torch.empty((cap, 4), dtype=torch.int32, pin_memory=True)


def pack_interactions(users, items, ratings, device) -> torch.Tensor:
    """(uid, iid, rating) columns -> int32 [n,4] ure_inter_t records on `device`.

    rating is cast the way RatingData does (reference read.py:113,124): float32(float64).  On a CUDA
    device the records are written straight into a pinned staging buffer and copied asynchronously.
    """
    n = len(users)
    cuda = torch.device(device).type == "cuda"
    stage = _staging(n) if cuda and n > 0 else torch.empty((max(n, 1), 4), dtype=torch.int32)
    rec = stage.numpy()[:n]
    users, items, ratings = np.asarray(users), np.asarray(items), np.asarray(ratings, dtype=np.float64)

    def fill(lo, hi):                                   # NumPy converts int64 / float64 -> int32 on assignment
        rec[lo:hi, 0] = users[lo:hi]
        rec[lo:hi, 1] = items[lo:hi]
        rec[lo:hi, 2].view(np.float32)[...] = ratings[lo:hi]
        rec[lo:hi, 3] = 0

    if n >= (1 << 17):                                  # the casts release the GIL: pack in parallel
        step = -(-n // _PACK_THREADS)
        list(_pack_pool().map(lambda lo: fill(lo, min(n, lo + step)), range(0, n, step)))
    else:
        fill(0, n)
    if not cuda:
        return stage[:n].clone()
    out = torch.empty((n, 4), dtype=torch.int32, device=device)
    if n > 0:
        out.copy_(stage[:n], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        _PINNED[stage.shape[0]].append((stage, ev))      # reusable once the copy has completed
    return out


_PINNED_BYTES = {}   # capacity -> list of (pinned uint8 buffer, event): staging for raw float64 uploads


def _staging_bytes(nbytes: int) -> torch.Tensor:
    cap = 1 << max(12, int(nbytes - 1).bit_length())
    pool = _PINNED_BYTES.setdefault(cap, [])
    for idx, item in enumerate(pool):
        if item[1] is None or item[1].query():
            del pool[idx]                # by position: list.remove(item) compares item with every entry before it, and
            return item[0]               # (tensor, event) == (other tensor, event) is an element-wise tensor comparison
    return torch.empty(cap, dtype=torch.uint8, pin_memory=True)


UPLOAD_RING_BYTES = 64 << 20         # segment of the two-segment staging ring of very large uploads
UPLOAD_ONE_SHOT_BYTES = 1 << 30      # uploads up to this size are staged whole (one pinned buffer, one DMA per array)


def _upload_ring(dst_ptr: int, src_ptr: int, nb: int) -> None:
    """Pageable host bytes [src, src + nb) -> device [dst, dst + nb) on the current stream through TWO page-locked
    segments of UPLOAD_RING_BYTES: the pool threads fill one (non-temporal stores) while the DMA engine drains the
    other, so the page-locked footprint of an upload does not grow with its size (a C4-sized rating table is 24 GB)."""
    L, seg, CH = _lib.lib(), int(UPLOAD_RING_BYTES), 1 << 21
    bufs = [_staging_bytes(seg), _staging_bytes(seg)]
    evs = [None, None]
    for k, lo in enumerate(range(0, nb, seg)):
        b, n = k & 1, min(seg, nb - lo)
        if evs[b] is not None:
            evs[b].synchronize()                                   # the DMA that last read this segment is done
        base = bufs[b].data_ptr()
        futs = [_pack_pool().submit(L.ure_host_stage_copy, C.c_void_p(base + o), C.c_void_p(src_ptr + lo + o), min(CH, n - o))
                for o in range(0, n, CH)]
        for f in futs:
            check(f.result(), "ure_host_stage_copy")
        check(L.ure_copy_to_device_async(C.c_void_p(dst_ptr + lo), C.c_void_p(base), n, _stream()), "ure_copy_to_device_async")
        evs[b] = torch.cuda.Event()
        evs[b].record()
    for b in range(2):
        _PINNED_BYTES.setdefault(bufs[b].shape[0], []).append((bufs[b], evs[b]))


def upload_interactions_many(raws, device, row_of: Optional[torch.Tensor] = None, defer: bool = False,
                             eager: Optional[list] = None):
    """float64 [3, n] arrays (uid, iid, rating/max_rating: what readRating returns, reference read.py:64-68) ->
    int32 [n,4] ure_inter_t records on `device`, packed ON the device (ure_pack_interactions_f64).

    The host only moves bytes: every array is copied into pinned staging memory (one thread per array, NumPy
    releases the GIL) and uploaded asynchronously; the casts of RatingData (read.py:111-113,124) and the optional
    user -> compact-row mapping (`row_of`, int32 device tensor) run in the pack kernel.

    defer=True returns (outs, finish): the staging copies are already running on the worker threads, `finish()`
    waits for them and queues the uploads + pack kernels -- the caller does other host work in between.
    eager[j] = (device columns, event) of an array whose copy was started earlier (eager_upload): only its pack kernel
    is queued here, behind the event."""
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("ultrare_b200: interactions are packed on a CUDA device (no CPU path exists)")
    arrs = []
    for raw in raws:
        raw = np.asarray(raw)
        if raw.ndim != 2 or raw.dtype != np.float64 or raw.shape[0] != 3:
            raw = np.ascontiguousarray(np.asarray(raw).reshape(3, -1)[:3], dtype=np.float64)
        arrs.append(raw)
    ns = [a.shape[1] for a in arrs]
    n_tot = sum(ns)
    out_all = torch.empty((n_tot, 4), dtype=torch.int32, device=dev)
    offs = np.concatenate([[0], np.cumsum(ns)]).astype(np.int64)
    outs = [out_all[offs[j]:offs[j + 1]] for j in range(len(arrs))]
    if n_tot == 0:
        return (outs, lambda: None) if defer else outs
    # ONE pinned staging buffer and ONE device buffer for all arrays; array j starts at a 64-byte boundary
    starts = np.zeros(len(arrs) + 1, dtype=np.int64)              # in doubles
    for j, n in enumerate(ns):
        starts[j + 1] = (starts[j] + 3 * n + 7) // 8 * 8
    tot_d = int(starts[-1])
    L = _lib.lib()
    if 8 * tot_d > UPLOAD_ONE_SHOT_BYTES:
        # too large to stage whole: array after array, each through the two-segment ring (or straight from its own
        # page-locked memory) into a device buffer that lives until its pack kernel has run

        def one_by_one():
            with torch.cuda.device(dev):
                for j in range(len(arrs)):
                    if not ns[j]:
                        continue
                    if eager is not None and eager[j] is not None:
                        cols_j, ev_j = eager[j]
                        cur = torch.cuda.current_stream()
                        cur.wait_event(ev_j)
                        cols_j.record_stream(cur)
                    else:
                        a = np.ascontiguousarray(arrs[j])
                        cols_j = torch.empty(3 * ns[j], dtype=torch.float64, device=dev)
                        if _is_page_locked(a):
                            check(L.ure_copy_to_device_async(C.c_void_p(cols_j.data_ptr()), C.c_void_p(int(a.ctypes.data)),
                                                             a.nbytes, _stream()), "ure_copy_to_device_async")
                        else:
                            _upload_ring(cols_j.data_ptr(), int(a.ctypes.data), a.nbytes)
                    check(L.ure_pack_interactions_f64(C.c_void_p(cols_j.data_ptr()), ns[j], ns[j], _ptr(row_of),
                                                      0 if row_of is None else int(row_of.shape[0]), _ptr(outs[j]), _stream()),
                          "ure_pack_interactions_f64")
                    del cols_j                                     # stream-ordered: the block is reused behind the pack kernel

        if defer:
            return outs, one_by_one
        one_by_one()
        return outs
    stage = _staging_bytes(8 * tot_d)
    stage_f = stage[:8 * tot_d].view(torch.float64)
    base = stage.data_ptr()
    cols_all = torch.empty(tot_d, dtype=torch.float64, device=dev)
    CHUNK = int(float(__import__('os').environ.get('URE_PACK_CHUNK_MB', '2')) * (1 << 20)) // 64 * 64   # bytes per staging task

    def fill(j, lo, hi):                                          # bytes [lo, hi) of array j, non-temporal stores
        check(L.ure_host_stage_copy(C.c_void_p(base + 8 * int(starts[j]) + lo), C.c_void_p(arrs[j].ctypes.data + lo),
                                    hi - lo), "ure_host_stage_copy")

    def ship(j):                                                  # main thread: async H2D + pack kernel of array j
        if eager is not None and eager[j] is not None:            # already on its way (or there): pack behind its event
            cols_j, ev_j = eager[j]
            cur = torch.cuda.current_stream()
            cur.wait_event(ev_j)
            cols_j.record_stream(cur)
            check(L.ure_pack_interactions_f64(C.c_void_p(cols_j.data_ptr()), ns[j], ns[j], _ptr(row_of),
                                              0 if row_of is None else int(row_of.shape[0]), _ptr(outs[j]), _stream()),
                  "ure_pack_interactions_f64")
            return
        lo, hi = int(starts[j]), int(starts[j]) + 3 * ns[j]
        src = base + 8 * lo if pinned[j] is None else int(arrs[j].ctypes.data)      # both page-locked
        check(L.ure_copy_to_device_async(C.c_void_p(cols_all.data_ptr() + 8 * lo), C.c_void_p(src), 8 * (hi - lo), _stream()),
              "ure_copy_to_device_async")
        check(L.ure_pack_interactions_f64(C.c_void_p(cols_all.data_ptr() + 8 * lo), ns[j], ns[j], _ptr(row_of),
                                          0 if row_of is None else int(row_of.shape[0]), _ptr(outs[j]), _stream()),
              "ure_pack_interactions_f64")

    todo = [j for j in range(len(arrs)) if ns[j]]
    pinned = [None] * len(arrs)           # arrays that already live in page-locked memory are uploaded from there
    for j in todo:
        if not arrs[j].flags.c_contiguous:
            arrs[j] = np.ascontiguousarray(arrs[j])
        if (eager is not None and eager[j] is not None) or _is_page_locked(arrs[j]):
            pinned[j] = True
    # arrays that already live in page-locked memory need no staging copy: their upload + pack are queued right here
    # (defer or not), so the DMA engine starts while the caller still does its host-side set-up
    shipped = set()
    with torch.cuda.device(dev):
        for j in todo:
            if pinned[j] is not None:
                ship(j)
                shipped.add(j)
    futs = None
    if n_tot >= (1 << 16):
        # staging copies on worker threads (ctypes releases the GIL); every array is shipped as soon as ITS
        # chunks are done, so the DMA engine works while the other arrays are still being copied
        futs = {j: [_pack_pool().submit(fill, j, lo, min(24 * ns[j], lo + CHUNK))
                    for lo in range(0, 24 * ns[j], CHUNK)] if pinned[j] is None else [] for j in todo}

    def finish():
        with torch.cuda.device(dev):
            for j in todo:
                if j in shipped:
                    continue
                if futs is None:
                    fill(j, 0, 24 * ns[j])
                else:
                    for f in futs[j]:
                        f.result()
                ship(j)
            ev = torch.cuda.Event()
            ev.record()
            _PINNED_BYTES[stage.shape[0]].append((stage, ev))

    if defer:
        return outs, finish
    finish()
    return outs


_PAGE_LOCKED = []        # (first byte, one past the last, weak reference to the owning tensor) of pinned_copy's buffers


def pinned_copy(a: np.ndarray) -> np.ndarray:
    """Copy of `a` in page-locked host memory (a NumPy view of a pinned torch tensor): arrays handed to
    RatingData / upload_interactions in this form are uploaded without the staging copy."""
    import weakref
    t = torch.empty(a.shape, dtype=_TORCH_DTYPE[a.dtype.name], pin_memory=True)
    out = t.numpy()
    out[...] = a
    _PAGE_LOCKED[:] = [e for e in _PAGE_LOCKED if e[2]() is not None]
    _PAGE_LOCKED.append((t.data_ptr(), t.data_ptr() + t.numel() * t.element_size(), weakref.ref(t)))
    return out


def _is_page_locked(arr: np.ndarray) -> bool:
    """Does the array live in page-locked memory?  Buffers of pinned_copy are known by address (no driver call per
    upload); anything else is asked through torch once."""
    p0 = int(arr.ctypes.data)
    p1 = p0 + arr.nbytes
    for lo, hi, ref in _PAGE_LOCKED:
        if lo <= p0 and p1 <= hi and ref() is not None:
            return True
    if not arr.flags.writeable:
        return False
    try:
        return bool(torch.from_numpy(arr).is_pinned())
    except Exception:
        return False


def upload_interactions(raw, device, row_of: Optional[torch.Tensor] = None, eager=None) -> torch.Tensor:
    """One array through upload_interactions_many."""
    return upload_interactions_many([raw], device, row_of, eager=None if eager is None else [eager])[0]


EAGER_MIN_ROWS = 1 << 16      # smaller arrays are not worth a stream hand-over


def eager_upload(raw, device):
    """Start the host -> device copy of a float64 [3, n] array that lives in page-locked memory RIGHT NOW, on the side
    stream (read.EAGER_UPLOAD_DEVICE: RatingData calls this from its constructor, so the bytes travel while the caller
    is still building loaders, routing deletions, laying out the batch).  Returns (device columns, event) -- what
    upload_interactions_many(eager=...) packs from -- or None when the array does not qualify."""
    if not (isinstance(raw, np.ndarray) and raw.dtype == np.float64 and raw.ndim == 2 and raw.shape[0] == 3 and
            raw.flags.c_contiguous and raw.shape[1] >= EAGER_MIN_ROWS and _is_page_locked(raw)):
        return None
    dev = torch.device(device)
    side = side_stream(dev)
    with torch.cuda.device(dev):
        with torch.cuda.stream(side):                  # the buffer comes from the side stream's pool
            cols = torch.empty(3 * raw.shape[1], dtype=torch.float64, device=dev)
        check(_lib.lib().ure_copy_to_device_async(C.c_void_p(cols.data_ptr()), C.c_void_p(int(raw.ctypes.data)), raw.nbytes,
                                                  C.c_void_p(side.cuda_stream)), "ure_copy_to_device_async")
        ev = torch.cuda.Event()
        ev.record(side)
    return cols, ev


_TORCH_DTYPE = {"uint8": torch.uint8, "int32": torch.int32, "int64": torch.int64, "float32": torch.float32,
                "float64": torch.float64, "int16": torch.int16}


def upload_array(a: np.ndarray, device, side: bool = False) -> torch.Tensor:
    """Small host array -> device through the pinned staging pool (asynchronous: the host does not wait for the
    work already queued on the stream, unlike a pageable .to(device)).  side: the copy runs on the upload side stream
    and the caller's stream waits for its event -- a table queued while a long kernel runs is resident when it ends."""
    a = np.ascontiguousarray(a)
    if side and SIDE_SMALL_UPLOADS and a.size:
        with on_side(device) as main:
            out = upload_array(a, device)
            out.record_stream(main)
        return out
    out = torch.empty(a.shape, dtype=_TORCH_DTYPE[a.dtype.name], device=device)
    if a.size == 0:
        return out
    stage = _staging_bytes(a.nbytes)
    stage.numpy()[:a.nbytes] = a.reshape(-1).view(np.uint8)
    with torch.cuda.device(device):
        out.view(-1).view(torch.uint8).copy_(stage[:a.nbytes], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        _PINNED_BYTES[stage.shape[0]].append((stage, ev))
    return out


def upload_table(a: np.ndarray, device) -> torch.Tensor:
    """Large host array -> device: staging copies in 2 MB tasks on the pack pool (non-temporal stores), one DMA; beyond
    UPLOAD_ONE_SHOT_BYTES through a two-segment staging ring (_upload_ring)."""
    a = np.ascontiguousarray(a)
    out = torch.empty(a.shape, dtype=_TORCH_DTYPE[a.dtype.name], device=device)
    nb = a.nbytes
    if nb < (1 << 21):
        return upload_array(a, device)
    if nb > UPLOAD_ONE_SHOT_BYTES:
        with torch.cuda.device(device):
            _upload_ring(out.data_ptr(), int(a.ctypes.data), nb)
        return out
    stage = _staging_bytes(nb)
    base, src, L, CHUNK = stage.data_ptr(), a.ctypes.data, _lib.lib(), 1 << 21
    futs = [_pack_pool().submit(L.ure_host_stage_copy, C.c_void_p(base + lo), C.c_void_p(src + lo), min(CHUNK, nb - lo))
            for lo in range(0, nb, CHUNK)]
    for f in futs:
        check(f.result(), "ure_host_stage_copy")
    with torch.cuda.device(device):
        out.view(-1).view(torch.uint8).copy_(stage[:nb], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        _PINNED_BYTES[stage.shape[0]].append((stage, ev))
    return out


def deletion_lists(pairs, n_map: int, device=None):
    """The per-user deleted-item CSR of ure_partition_interactions_del, built on the device by ure_seen_lists:
    (off int64 [n_map + 1], items int32 ascending within each user), or None when no pair can match a row.
    `pairs`: array-like [n, >= 2] of (user, item) ids on the host, or such a CUDA tensor; further columns are ignored
    and the ids are truncated to integers, as the partition truncates the table's.  Negative ids raise ValueError;
    pairs whose user lies outside [0, n_map) cannot match a kept row and are dropped.  Host pairs are checked on the
    host and uploaded once; device pairs are checked on the device (one synchronisation)."""
    on_dev = isinstance(pairs, torch.Tensor)
    p = pairs if on_dev else np.asarray(pairs)
    if len(p) == 0:
        return None
    if p.ndim != 2 or p.shape[1] < 2:
        raise ValueError(f"deletion_lists: pairs must be [n, >= 2], got {tuple(p.shape)}")
    if on_dev:
        _need_cuda(p)
        p = p[:, :2].to(torch.int64)
    else:
        p = p[:, :2].astype(np.int64)
    if bool((p < 0).any()):
        raise ValueError("deletion_lists: user and item ids must be non-negative")
    if bool((p[:, 1] >= 2 ** 31).any()):
        raise ValueError("deletion_lists: item ids must be below 2^31")
    p = p[p[:, 0] < n_map]
    if p.shape[0] == 0:
        return None
    n_item = int(p[:, 1].max()) + 1
    if on_dev:
        rec = torch.zeros((p.shape[0], 4), dtype=torch.int32, device=p.device)
        rec[:, :2] = p.to(torch.int32)
    else:
        rec = np.zeros((p.shape[0], 4), dtype=np.int32)
        rec[:, :2] = p
        rec = upload_array(rec, torch.device('cuda' if device is None else device))
    return seen_lists(rec, int(n_map), n_item)


def partition_interactions(table: torch.Tensor, max_rating: float, owner: torch.Tensor,
                           deleted: Optional[torch.Tensor], n_shards: int, columns: bool = True, del_lists=None):
    """readRating's filter + split on the device (ure_partition_interactions).  table: float64 [3,n] (columns=True)
    or [n,3] (rows of the CSV, columns=False); owner int32 [n_map]; deleted uint8 [n_map] or None; del_lists: the
    deleted ratings as deletion_lists(pairs, n_map) returns them, or None (ure_partition_interactions_del drops every
    row whose (user, item) is listed).  Returns (records int32 [n,4] whose first shard_off[-1] rows are the shards'
    runs back to back, shard_off int64 device tensor [n_shards+1])."""
    _need_cuda(table, owner, deleted)
    assert table.dtype == torch.float64 and table.dim() == 2 and table.is_contiguous()
    assert owner.dtype == torch.int32 and (deleted is None or (deleted.dtype == torch.uint8 and deleted.shape == owner.shape))
    if del_lists is not None:
        del_off, del_item = del_lists
        _need_cuda(del_off, del_item)
        assert del_off.dtype == torch.int64 and del_off.shape == (owner.shape[0] + 1,) and del_off.is_contiguous()
        assert del_item.dtype == torch.int32 and del_item.is_contiguous() and del_item.device == table.device
    if columns:
        assert table.shape[0] == 3
        n, rs, cs = table.shape[1], 1, max(1, table.shape[1])
    else:
        assert table.shape[1] == 3
        n, rs, cs = table.shape[0], 3, 1
    L = _lib.lib()
    out = torch.empty((n, 4), dtype=torch.int32, device=table.device)
    off = torch.empty(n_shards + 1, dtype=torch.int64, device=table.device)
    hist = torch.empty((L.ure_partition_blocks(), 256), dtype=torch.int32, device=table.device)
    with torch.cuda.device(table.device):
        if del_lists is None:
            check(L.ure_partition_interactions(_ptr(table), n, rs, cs, float(max_rating), _ptr(owner), _ptr(deleted),
                                               owner.shape[0], n_shards, _ptr(out), _ptr(hist), _ptr(off), _stream()),
                  "ure_partition_interactions")
        else:
            check(L.ure_partition_interactions_del(_ptr(table), n, rs, cs, float(max_rating), _ptr(owner), _ptr(deleted),
                                                   owner.shape[0], n_shards, _ptr(del_off), _ptr(del_item), _ptr(out),
                                                   _ptr(hist), _ptr(off), _stream()),
                  "ure_partition_interactions_del")
    return out, off


def remap_users(inter: torch.Tensor, row_of: torch.Tensor) -> torch.Tensor:
    """Copy of `inter` whose user field is row_of[user] (ure_remap_users)."""
    _need_cuda(inter, row_of)
    assert inter.dtype == torch.int32 and inter.is_contiguous() and row_of.dtype == torch.int32
    out = torch.empty_like(inter)
    with torch.cuda.device(inter.device):
        check(_lib.lib().ure_remap_users(_ptr(inter), inter.shape[0], _ptr(row_of), row_of.shape[0], _ptr(out), _stream()),
              "ure_remap_users")
    return out


def download_many(tensors: Sequence[torch.Tensor], copy: bool = True) -> List[np.ndarray]:
    """Device tensors -> host arrays through ONE pinned staging buffer and ONE synchronisation (a `.cpu()` per
    tensor is a pageable copy + a synchronisation each).  Tensors that lie back to back in device memory (the tables
    of a batch arena) travel as one transfer.  copy=False: the arrays are views of a page-locked buffer of their own
    (no second pass over the bytes on the host); it stays alive as long as any of them does."""
    if not tensors:
        return []
    dev = tensors[0].device
    tensors = [t.contiguous() for t in tensors]
    sizes = [t.numel() * t.element_size() for t in tensors]
    offs, runs, o = [], [], 0                # runs: (device address, staging offset, bytes) of every transfer
    for t, b in zip(tensors, sizes):
        if runs and b and t.data_ptr() == runs[-1][0] + runs[-1][2]:
            offs.append(runs[-1][1] + runs[-1][2])
            runs[-1] = (runs[-1][0], runs[-1][1], runs[-1][2] + b)
            o = runs[-1][1] + runs[-1][2]
        else:
            o = (o + 63) // 64 * 64
            offs.append(o)
            if b:
                runs.append((t.data_ptr(), o, b))
            o += b
    total = o + 64
    stage = _staging_bytes(total) if copy else torch.empty(total, dtype=torch.uint8, pin_memory=True)
    with torch.cuda.device(dev):
        for src, so, b in runs:         # raw async copies: a torch copy_ per tensor costs ~20 us of dispatch each
            check(_lib.lib().ure_copy_to_host_async(C.c_void_p(stage.data_ptr() + so), C.c_void_p(src), b, _stream()),
                  "ure_copy_to_host_async")
        ev = torch.cuda.Event()
        ev.record()
        ev.synchronize()
    host = stage.numpy()
    outs = [host[int(o_):int(o_) + b].view(np.dtype(str(t.dtype).replace("torch.", ""))).reshape(tuple(t.shape))
            for t, o_, b in zip(tensors, offs, sizes)]
    if copy:
        outs = [x.copy() for x in outs]
        _PINNED_BYTES.setdefault(stage.shape[0], []).append((stage, None))
    return outs


def pointer_table(tensors: Sequence[torch.Tensor], device) -> torch.Tensor:
    return upload_array(np.array([t.data_ptr() for t in tensors], dtype=np.int64), device, side=True)


# ------------------------------------------------------------------------------ MF training
OWNER_SCHED_BYTES = 512 << 20  # device memory one ShardBatch may spend on owner-mode schedule tables
RUNS_LIST_BYTES = 2 << 30      # device memory one ShardBatch may spend on the RUNS schedule's step lists
OWNER_FORCE = None             # test hook: (owner_flags, list_cap) the owner schedule must use
DEFAULT_MF_MODE = "auto"       # schedule ShardBatch picks when the caller does not say (see ShardBatch)


class ShardState:
    """Device state of one shard model: what Scratch.train builds (scratch.py:59,65-69)."""

    def __init__(self, inter: torch.Tensor, P: torch.Tensor, Q: torch.Tensor, epochs: int,
                 shard_id: int = 0, perm_seed: int = 42, perm: Optional[torch.Tensor] = None, scratch=None):
        """scratch: optional (bufP, bufQ, gP, gQ, sse) zero-filled views of a batch allocation."""
        _need_cuda(inter, P, Q, perm)
        assert inter.dtype == torch.int32 and inter.dim() == 2 and inter.shape[1] == 4
        assert P.dtype == torch.float32 and Q.dtype == torch.float32 and P.shape[1] == Q.shape[1]
        self.inter, self.P, self.Q = inter.contiguous(), P, Q
        assert P.is_contiguous() and Q.is_contiguous()
        if scratch is None:
            self.bufP, self.bufQ = torch.zeros_like(P), torch.zeros_like(Q)
            self.gP, self.gQ = torch.zeros_like(P), torch.zeros_like(Q)
            self.sse = torch.zeros(max(1, epochs), dtype=torch.float64, device=P.device)
        else:
            self.bufP, self.bufQ, self.gP, self.gQ, self.sse = scratch
        self.perm = None
        if perm is not None:
            assert perm.dtype == torch.int32 and perm.shape == (epochs, inter.shape[0])
            self.perm = perm.contiguous()
        self.n = int(inter.shape[0])
        self.shard_id, self.perm_seed, self.epochs = int(shard_id), int(perm_seed) & 0xFFFFFFFF, int(epochs)
        self.group = 0
        self.lastP = self.lastQ = self.touched = None          # lazy mode state (ShardBatch(mode="lazy"))
        self.inter_u = self.inter_i = self.off_u = self.off_i = self.perm_inv = None   # owner mode state
        self.tmp_u = self.tmp_i = None

    def descriptor(self) -> MFShard:
        d = MFShard()
        d.inter, d.perm = self.inter.data_ptr(), (self.perm.data_ptr() if self.perm is not None else None)
        d.P, d.Q = self.P.data_ptr(), self.Q.data_ptr()
        d.bufP, d.bufQ = self.bufP.data_ptr(), self.bufQ.data_ptr()
        d.gP, d.gQ, d.sse = self.gP.data_ptr(), self.gQ.data_ptr(), self.sse.data_ptr()
        d.lastP = self.lastP.data_ptr() if self.lastP is not None else None
        d.lastQ = self.lastQ.data_ptr() if self.lastQ is not None else None
        d.touched = self.touched.data_ptr() if self.touched is not None else None
        for name in ("inter_u", "inter_i", "off_u", "off_i", "perm_inv", "tmp_u", "tmp_i"):
            t = getattr(self, name)
            setattr(d, name, t.data_ptr() if t is not None else None)
        d.n, d.n_user, d.n_item = self.n, self.P.shape[0], self.Q.shape[0]
        d.shard_id, d.perm_seed, d.group = self.shard_id, self.perm_seed, self.group
        return d

    def steps_per_epoch(self, batch: int) -> int:
        return -(-self.n // batch)


class ShardBatch:
    """All shard models a GPU owns, trained together by one persistent launch.

    mode: "dense" (L2-atomic scatter + dense sweep), "lazy" (closed-form catch-up of untouched rows),
    "owner" (owner-computes, weights resident in shared memory: small tables only) or "auto" = owner when
    its plan fits the shared memory of the SMs, else dense.  The three schedules compute the same update."""

    def __init__(self, shards: List[ShardState], d: int, batch: int, lr: float = 1e-3, lr_decay: float = 0.95,
                 lr_step: int = 50, weight_decay: float = 0.1, momentum: float = 0.9, lazy: bool = False,
                 mode: Optional[str] = None, owner_cache: bool = True, after_prepare=None):
        """after_prepare: optional callable run once the set-up kernels that only read the records are queued
        (alloc_shard_batch(defer_init=True)'s fills), before the set-up waits for the plan."""
        self._after_prepare = after_prepare
        if not 1 <= len(shards) <= _lib.URE_MAX_SHARDS:
            raise ValueError(f"1..{_lib.URE_MAX_SHARDS} shards per launch")
        mode = ("lazy" if lazy else DEFAULT_MF_MODE) if mode is None else mode
        if mode not in ("dense", "lazy", "owner", "auto", "runs"):
            raise ValueError(f"mode {mode!r}")
        self.shards = shards
        self.n_shards = len(shards)
        self.device = shards[0].P.device
        self.epochs = shards[0].epochs
        assert all(s.epochs == self.epochs for s in shards)
        self.total_steps = max(s.steps_per_epoch(batch) for s in shards) * self.epochs
        self.ws = torch.zeros(int(_lib.lib().ure_mf_train_workspace_bytes()), dtype=torch.uint8, device=self.device)
        self.hp = MFHParams(d=d, batch=batch, lr0=lr, lr_decay=lr_decay, lr_step=lr_step,
                            weight_decay=weight_decay, momentum=momentum, mode=_lib.MF_DENSE,
                            decay=None, decay_len=0, owner_cap_rows=0, owner_cap_slots=0, owner_flags=0,
                            owner_spe_cap=0, owner_sched_rows=0, owner_sched=None, owner_sched_off=None,
                            owner_sched_step0=0, owner_sched_stride=0)
        self.owner_plan = None
        self.launches_per_pass = 0          # kernels of ours this batch has launched (set-up + schedule + training)
        self._owner_cache = bool(owner_cache)       # False: keep the records in L2 (tests of the uncached variant)
        self.warps_group0 = self._split_groups(shards)   # before the first table upload: descriptors are final
        if mode in ("owner", "auto"):
            mode = self._prepare_owner(mode == "owner")
        self.mode = mode
        self._run_after_prepare()          # schedules without a set-up pass: right away
        self.lazy = mode in ("lazy", "runs")            # rows catch up in closed form: flush() before reading P / Q
        self.decay = None
        if mode == "runs":
            self._prepare_runs(lr, weight_decay, momentum)
        elif self.lazy:
            # M^n for n = 0..total_steps (float64 on the host): the n-step gradient-free SGD update
            # [w;buf] <- M^n [w;buf], M = [[1-lr*wd, -lr*mu],[wd, mu]]  (csrc/mf_train_lazy.cu)
            M = np.array([[1.0 - lr * weight_decay, -lr * momentum], [weight_decay, momentum]])
            T = np.empty((self.total_steps + 2, 2, 2))
            T[0] = np.eye(2)
            for n in range(1, len(T)):
                T[n] = M @ T[n - 1]
            self.decay = torch.from_numpy(T.reshape(-1, 4).astype(np.float32)).to(self.device)
            for s in shards:
                s.lastP = torch.zeros(s.P.shape[0], dtype=torch.int32, device=self.device)
                s.lastQ = torch.zeros(s.Q.shape[0], dtype=torch.int32, device=self.device)
                s.touched = torch.zeros(4 * (1 + batch), dtype=torch.int32, device=self.device)
            self.hp.mode, self.hp.decay, self.hp.decay_len = _lib.MF_LAZY, self.decay.data_ptr(), len(self.decay)
        self._upload_table()
        self.step = 0

    def _run_after_prepare(self):
        hook, self._after_prepare = self._after_prepare, None
        if hook is not None:
            hook()

    def _upload_table(self):
        arr = (MFShard * len(self.shards))(*[s.descriptor() for s in self.shards])
        blob = bytes(arr)
        if getattr(self, "_table_blob", None) == blob:       # nothing changed since the last upload
            return
        self.host_table, self._table_blob = arr, blob
        self.table = upload_array(np.frombuffer(blob, dtype=np.uint8), self.device)

    def _prepare_owner(self, required: bool) -> str:
        """Owner-mode set-up: one allocation for the sorted record copies + row offsets of every shard,
        ure_mf_owner_prepare (counting sorts + CTA plan), one 16-byte read-back of the plan."""
        L = _lib.lib()
        shards, dev = self.shards, self.device
        tq = [time.perf_counter()]
        if len(shards) > int(L.ure_mf_grid_size()):
            if required:
                raise RuntimeError("owner mode needs at most one shard per SM")
            return "dense"
        n_tot = sum(s.n for s in shards)
        # cheap refusal before any allocation: the weights + momentum of all rows must fit the SMs' shared memory
        state = sum(s.P.shape[0] + s.Q.shape[0] for s in shards) * 8 * self.hp.d
        if state > int(L.ure_mf_grid_size()) * (200 << 10) or n_tot >= (1 << 31):
            if required:
                raise RuntimeError(f"owner mode does not fit this problem: {state} bytes of row state")
            return "dense"
        rec = torch.empty((4, max(1, n_tot), 4), dtype=torch.int32, device=dev)      # sorted copies + radix scratch
        n_off = sum(s.P.shape[0] + s.Q.shape[0] + 4 for s in shards)
        off = torch.zeros(n_off, dtype=torch.int32, device=dev)
        o = r = 0
        for s in shards:
            s.inter_u, s.inter_i = rec[0, r:r + s.n], rec[1, r:r + s.n]
            s.tmp_u, s.tmp_i = rec[2, r:r + s.n], rec[3, r:r + s.n]
            r += s.n
            nu, ni = s.P.shape[0] + 2, s.Q.shape[0] + 2
            s.off_u, s.off_i = off[o:o + nu], off[o + nu:o + nu + ni]
            o += nu + ni
            s.perm_inv = torch.empty_like(s.perm) if s.perm is not None else None
        radix = torch.empty(int(L.ure_mf_owner_radix_bytes(len(shards))) // 4, dtype=torch.int32, device=dev)
        self._owner_keep = (rec, off, radix)
        tq.append(time.perf_counter())
        self._upload_table()
        tq.append(time.perf_counter())
        max_rows = max(max(s.P.shape[0], s.Q.shape[0]) for s in shards)
        npass = 1
        while npass < 4 and (max_rows - 1) >> (8 * npass):
            npass += 1
        self.prepare_launches = 2 + 3 * npass + 1 + 1     # count + scan, radix passes, perm inverse, plan
        self.launches_per_pass += self.prepare_launches
        with torch.cuda.device(dev):
            check(L.ure_mf_owner_prepare(_ptr(self.table), len(shards), C.byref(self.hp), self.epochs, int(max_rows),
                                         _ptr(radix), _ptr(self.ws), _stream()), "ure_mf_owner_prepare")
        rb = self.ws[:16].clone()                      # the plan, snapshotted before anything else is queued
        self._run_after_prepare()
        t0 = time.perf_counter()
        max_rows, max_slots, max_spe, avail = rb.view(torch.int32).tolist()             # the one sync of the set-up
        self.plan_sync_ms = (time.perf_counter() - t0) * 1e3          # host wait for upload + sorts (diagnostics)
        tq += [t0, time.perf_counter()]
        cap_rows, cap_slots, spe_cap = max(1, max_rows), max(16, -(-max_slots // 16) * 16), max(1, max_spe)
        d = self.hp.d

        def need_of(cap_list, flags):
            return int(L.ure_mf_owner_smem_bytes(d, cap_rows, cap_slots, cap_list, spe_cap, flags))

        # shared-memory configurations, fastest first: record cache (every owned slot's record resident); batch
        # lists and their records staged per step, as many entries as fit (a longer list is read from the schedule
        # table); the same with the schedule pre-pass running without its record-index cache
        cands = []
        if self._owner_cache and max(max(s.P.shape[0], s.Q.shape[0]) for s in shards) <= (1 << 20):
            cands.append((1, cap_slots))
        for f in (0, 2):
            need16 = need_of(16, f)
            if need16 <= avail:                         # 10 bytes of shared memory per staged entry
                cands.append((f, min(cap_slots, 16 + (avail - need16) // 160 * 16)))
        if OWNER_FORCE is not None:                      # tests: (flags, list_cap) instead of the fastest that fits
            cands = [(OWNER_FORCE[0], min(cap_slots, max(16, OWNER_FORCE[1] // 16 * 16)))]
        pick = next(((f, c) for f, c in cands if need_of(c, f) <= avail and
                     (c >= min(cap_slots, 1024) or OWNER_FORCE is not None)), None)
        fits = pick is not None and cap_slots <= 65520 and cap_rows < 4096 and max_spe <= 8192
        flags, cap_list = pick if pick is not None else (0, cap_slots)
        cached = bool(flags & 1)
        self.owner_plan = {"smem_need": need_of(cap_list, flags), "smem_need_cached": need_of(cap_slots, 1),
                           "smem_avail": avail, "cached": cached, "flags": flags, "list_cap": cap_list,
                           "max_rows_per_cta": max_rows, "max_slots_per_cta": max_slots, "max_steps_per_epoch": max_spe}
        if not fits:
            if required:
                raise RuntimeError(f"owner mode does not fit this problem: {self.owner_plan}")
            for s in shards:
                s.inter_u = s.inter_i = s.off_u = s.off_i = s.perm_inv = s.tmp_u = s.tmp_i = None
            self._owner_keep = None
            return "dense"
        # schedule tables (ure_mf_owner_schedule): as many epochs per shard as OWNER_SCHED_BYTES allows, >= 2
        grid = int(L.ure_mf_grid_size())
        stride = max(1, 2 * n_tot)
        row_bytes = 2 * stride + 4 * grid * (spe_cap + 1)
        n_rows = int(min(self.epochs + 1, max(2, OWNER_SCHED_BYTES // row_bytes)))
        self._sched = torch.empty((n_rows, stride), dtype=torch.int16, device=dev)
        self._sched_off = torch.empty((n_rows, grid, spe_cap + 1), dtype=torch.int32, device=dev)
        self._sched_cover = (0, 0)                     # global steps [a, b) the tables are valid for
        self._spes = [s.steps_per_epoch(self.hp.batch) for s in shards if s.n > 0]
        self.owner_plan["schedule_rows"], self.owner_plan["schedule_bytes"] = n_rows, n_rows * row_bytes
        self.hp.mode = _lib.MF_OWNER
        self.hp.owner_cap_rows, self.hp.owner_cap_slots, self.hp.owner_spe_cap = cap_rows, cap_slots, spe_cap
        self.hp.owner_flags, self.hp.owner_cap_list = int(flags), int(cap_list)
        self.hp.owner_max_n = max(s.n for s in shards)
        self.hp.owner_sched, self.hp.owner_sched_off = self._sched.data_ptr(), self._sched_off.data_ptr()
        self.hp.owner_sched_rows, self.hp.owner_sched_stride, self.hp.owner_sched_step0 = n_rows, stride, 0
        tq.append(time.perf_counter())
        self.prepare_ms = dict(zip(("alloc", "table", "launch", "sync", "plan+sched_alloc"),
                                   (np.diff(tq) * 1e3).round(3).tolist()))
        return "owner"

    def _decay_table(self, lr, weight_decay, momentum):
        """M^n for n = 0..total_steps (float64 on the host): the n-step gradient-free SGD update
        [w;buf] <- M^n [w;buf], M = [[1-lr*wd, -lr*mu],[wd, mu]]  (csrc/mf_train_lazy.cu, mf_train_runs.cu)"""
        M = np.array([[1.0 - lr * weight_decay, -lr * momentum], [weight_decay, momentum]])
        T = np.empty((self.total_steps + 2, 2, 2))
        T[0] = np.eye(2)
        for n in range(1, len(T)):
            T[n] = M @ T[n - 1]
        return torch.from_numpy(T.reshape(-1, 4).astype(np.float32)).to(self.device)

    def _prepare_runs(self, lr, weight_decay, momentum):
        """RUNS schedule set-up (csrc/mf_train_runs.cu): the user-sorted / item-sorted record copies of the owner
        set-up, two row slots + a version tag per row, step lists for a window of epochs, the M^n table."""
        L = _lib.lib()
        shards, dev, d, K = self.shards, self.device, self.hp.d, len(self.shards)
        n_tot = sum(s.n for s in shards)
        max_n = max(s.n for s in shards)
        spe_cap = max(1, max(s.steps_per_epoch(self.hp.batch) for s in shards))
        if spe_cap >= 1024:
            raise RuntimeError(f"runs mode handles < 1024 steps per epoch ({spe_cap})")
        rec = torch.empty((2, max(1, n_tot), 4), dtype=torch.int32, device=dev)
        tmp = torch.empty((2, max(1, n_tot), 4), dtype=torch.int32, device=dev)       # radix scratch: freed below
        n_off = sum(s.P.shape[0] + s.Q.shape[0] + 4 for s in shards)
        off = torch.zeros(n_off, dtype=torch.int32, device=dev)
        rows = int(min(self.epochs, max(1, RUNS_LIST_BYTES // max(1, 8 * n_tot))))
        lists = torch.empty((2, rows * max(1, n_tot)), dtype=torch.int32, device=dev)
        loff = torch.zeros((K, 2, rows, spe_cap + 1), dtype=torch.int32, device=dev)
        keep, o, r, lo = [rec, off, lists, loff], 0, 0, 0
        runs = (_lib.MFRuns * K)()
        for j, s in enumerate(shards):
            s.inter_u, s.inter_i = rec[0, r:r + s.n], rec[1, r:r + s.n]
            s.tmp_u, s.tmp_i = tmp[0, r:r + s.n], tmp[1, r:r + s.n]
            r += s.n
            nu, ni = s.P.shape[0] + 2, s.Q.shape[0] + 2
            s.off_u, s.off_i = off[o:o + nu], off[o + nu:o + nu + ni]
            o += nu + ni
            s.perm_inv = torch.empty_like(s.perm) if s.perm is not None else None
            slotP = torch.empty((2, s.P.shape[0], 2 * d), dtype=torch.float32, device=dev)
            slotQ = torch.empty((2, s.Q.shape[0], 2 * d), dtype=torch.float32, device=dev)
            metaP = torch.empty(s.P.shape[0], dtype=torch.int64, device=dev)
            metaQ = torch.empty(s.Q.shape[0], dtype=torch.int64, device=dev)
            keep += [slotP, slotQ, metaP, metaQ]
            runs[j].slotP, runs[j].slotQ, runs[j].metaP, runs[j].metaQ = (t.data_ptr() for t in (slotP, slotQ, metaP, metaQ))
            runs[j].list_u = lists[0, lo:].data_ptr()
            runs[j].list_i = lists[1, lo:].data_ptr()
            lo += rows * s.n
            runs[j].loff_u, runs[j].loff_i = loff[j, 0].data_ptr(), loff[j, 1].data_ptr()
        radix = torch.empty(int(L.ure_mf_owner_radix_bytes(K)) // 4, dtype=torch.int32, device=dev)
        self._upload_table()
        max_rows = max(max(s.P.shape[0], s.Q.shape[0]) for s in shards)
        with torch.cuda.device(dev):
            check(L.ure_mf_owner_prepare(_ptr(self.table), K, C.byref(self.hp), self.epochs, int(max_rows), _ptr(radix),
                                         _ptr(self.ws), _stream()), "ure_mf_owner_prepare")
        del tmp, radix
        for s in shards:
            s.tmp_u = s.tmp_i = None
        self.decay = self._decay_table(lr, weight_decay, momentum)
        self._runs_table = upload_array(np.frombuffer(bytes(runs), dtype=np.uint8), dev)
        self._runs_scratch = torch.empty(int(L.ure_mf_runs_scratch_bytes(K, max_n, rows, spe_cap)), dtype=torch.uint8,
                                         device=dev)
        self._runs_keep, self._runs_max_n = keep, max_n
        self.hp.mode, self.hp.decay, self.hp.decay_len = _lib.MF_RUNS, self.decay.data_ptr(), len(self.decay)
        self.hp.runs, self.hp.runs_rows, self.hp.runs_spe_cap, self.hp.runs_step0 = self._runs_table.data_ptr(), rows, spe_cap, 0
        with torch.cuda.device(dev):
            check(L.ure_mf_runs_init(_ptr(self.table), K, C.byref(self.hp), _stream()), "ure_mf_runs_init")
        self._sched_cover = (0, 0)
        self._spes = [s.steps_per_epoch(self.hp.batch) for s in shards if s.n > 0]

    @staticmethod
    def _split_groups(shards, total_warps: int = 32, min_warps: int = 6) -> int:
        """Greedy split of the shards into two warp groups of near-equal interaction count; returns the
        number of warps of group 0 (32 = a single group)."""
        if len(shards) < 2:
            for s in shards:
                s.group = 0
            return total_warps
        load = [0, 0]
        for s in sorted(shards, key=lambda s: -s.n):
            g = 0 if load[0] <= load[1] else 1
            s.group = g
            load[g] += s.n
        w0 = int(round(total_warps * load[0] / max(1, load[0] + load[1])))
        return min(total_warps - min_warps, max(min_warps, w0))

    def train(self, step_end: Optional[int] = None) -> None:
        """Advance every shard to global step `step_end` (default: the end of training)."""
        step_end = self.total_steps if step_end is None else min(int(step_end), self.total_steps)
        if step_end <= self.step:
            return
        L = _lib.lib()
        with torch.cuda.device(self.device):
            while self.step < step_end:
                t1 = step_end
                if self.mode in ("owner", "runs"):
                    t1 = min(step_end, self._schedule_window())
                check(L.ure_mf_train(_ptr(self.table), self.n_shards, C.byref(self.hp), self.epochs,
                                     self.step, t1, self.warps_group0, _ptr(self.ws), _stream()), "ure_mf_train")
                self.launches_per_pass += 1
                self.step = t1

    def _schedule_window(self) -> int:
        """OWNER / RUNS: make sure the schedule tables cover self.step (queue the pre-pass if not); returns the global
        step the window ends at.  The tables hold `rows` epochs per shard from the window's first step on."""
        L = _lib.lib()
        a, b = self._sched_cover
        rows = self.hp.owner_sched_rows if self.mode == "owner" else self.hp.runs_rows
        if not (a <= self.step < b):
            with torch.cuda.device(self.device):
                if self.mode == "owner":
                    check(L.ure_mf_owner_schedule(_ptr(self.table), self.n_shards, C.byref(self.hp), self.epochs,
                                                  self.step, _stream()), "ure_mf_owner_schedule")
                    self.launches_per_pass += 1
                else:
                    check(L.ure_mf_runs_schedule(_ptr(self.table), self.n_shards, C.byref(self.hp), self.epochs,
                                                 self.step, self._runs_max_n, _ptr(self._runs_scratch), _stream()),
                          "ure_mf_runs_schedule")
                    self.launches_per_pass += 3
            a = self.step                  # shard s leaves the window at step (a // spe_s + rows) * spe_s
            b = min([(a // spe + rows) * spe for spe in self._spes
                     if a // spe + rows < self.epochs] or [self.total_steps])
            self._sched_cover = (a, b)
            if self.mode == "owner":
                self.hp.owner_sched_step0 = a
            else:
                self.hp.runs_step0 = a
        return b

    def reset_for_rerun(self) -> None:
        """Back to step 0 with zero momentum and losses (the weights stay): bench.py times the training launch alone."""
        for st in self.shards:
            st.bufP.zero_()
            st.bufQ.zero_()
            st.sse.zero_()
        self.step = 0

    def flush(self) -> None:
        """Lazy mode: advance every row to the current step (call before reading P / Q)."""
        if self.mode == "runs":
            with torch.cuda.device(self.device):
                check(_lib.lib().ure_mf_runs_flush(_ptr(self.table), self.n_shards, C.byref(self.hp), self.epochs,
                                                   self.step, _stream()), "ure_mf_runs_flush")
        elif self.lazy:
            with torch.cuda.device(self.device):
                check(_lib.lib().ure_mf_flush(self.host_table, len(self.shards), C.byref(self.hp), self.epochs,
                                              self.step, _stream()), "ure_mf_flush")

    def interactions_trained(self) -> int:
        return sum(s.n for s in self.shards) * self.epochs

    def train_losses_async(self):
        """train_losses without the wait: the D2H copies are queued behind the work already on the stream and the
        returned callable waits for them when the values are needed (the host keeps launching meanwhile)."""
        sse = self._sse_matrix()
        K, E = sse.shape
        nb = sse.numel() * 8
        owner = self.mode == "owner"
        host = _staging_bytes(nb + 64)
        with torch.cuda.device(sse.device):
            # on their own stream behind an event of the caller's: what the caller queues next (merge, evaluation)
            # does not wait for these two copies
            main = torch.cuda.current_stream(sse.device)
            back = side_stream(sse.device, 1)
            done = torch.cuda.Event()
            done.record(main)
            back.wait_event(done)
            sse.record_stream(back)
            if owner:
                self.ws.record_stream(back)
            with torch.cuda.stream(back):
                host[:nb].view(torch.float64).copy_(sse.view(-1), non_blocking=True)
                if owner:
                    host[nb:nb + 4].copy_(self.ws[16:20], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(back)
        ns = self._shard_sizes()

        def wait() -> List[np.ndarray]:
            ev.synchronize()
            vals = host[:nb].view(torch.float64).numpy().reshape(K, E).copy()
            err = int(host[nb:nb + 4].view(torch.int32).item()) if owner else 0
            _PINNED_BYTES.setdefault(host.shape[0], []).append((host, None))
            if err == 2:
                _PLAN_HINTS.pop(getattr(self, "_plan_sig", None), None)
                raise PlanHintMiss("ultrare_b200: the remembered owner plan does not cover this batch; repeat the pass")
            if err != 0:
                raise RuntimeError("ultrare_b200: owner schedule asked for a step outside its scheduled window")
            return [np.sqrt(vals[j] / ns[j]) for j in range(K)]
        return wait

    def _sse_matrix(self) -> torch.Tensor:
        return torch.stack([s.sse for s in self.shards])

    def _shard_sizes(self):
        return [max(1, s.n) for s in self.shards]

    def train_losses(self) -> List[np.ndarray]:
        """Per shard: sqrt(sse_epoch / n) for every epoch (utils.py:108).  Synchronises (one D2H)."""
        return self.train_losses_async()()


class ShardView:
    """One shard of an ArenaShardBatch: the tensors ShardState exposes, as views into the arena (made on demand)."""

    def __init__(self, inter, P, Q, bufP, bufQ, gP, gQ, sse, n, shard_id, perm_seed, epochs, perm=None):
        self.inter, self.P, self.Q, self.bufP, self.bufQ, self.gP, self.gQ, self.sse = inter, P, Q, bufP, bufQ, gP, gQ, sse
        self.n, self.shard_id, self.perm_seed, self.epochs, self.perm = n, shard_id, perm_seed, epochs, perm

    def steps_per_epoch(self, batch: int) -> int:
        return -(-self.n // batch)


class PlanHintMiss(RuntimeError):
    """An optimistic owner launch (capacities from an earlier plan of the same shapes) did not cover the plan the
    set-up kernels found: nothing was trained; the caller repeats the pass (the hint is gone, so it waits for the plan)."""


_PLAN_HINTS = {}          # batch signature -> (max_rows, max_slots, max_spe, smem) of the last plan read back
PLAN_HINT_MARGIN = 0.03   # capacities of an optimistic launch: the remembered maxima plus this fraction


class ArenaShardBatch(ShardBatch):
    """ShardBatch whose whole device state is ONE allocation laid out, described and prepared by the native runtime
    (csrc/mf_batch.cu: ure_mf_batch_layout / _setup / _plan): the host makes one allocation, one library call that
    queues the descriptor upload, the clears and the owner set-up kernels, one N(0, std) fill of the weights, and
    reads the 16-byte plan -- no per-shard tensors exist before the training launch is queued (the per-shard views
    of `shards` are built on first use, while the GPU trains).

    recs: per shard the device records (user field = row of the shard's table); rows_P: rows of every user table."""

    def __init__(self, recs, rows_P, n_item: int, d: int, batch: int, epochs: int, shard_ids, perm_seed: int = 42,
                 perms=None, lr: float = 1e-3, lr_decay: float = 0.95, lr_step: int = 50, weight_decay: float = 0.1,
                 momentum: float = 0.9, generator=None, std: float = 1.0, mode: str = "auto", owner_cache: bool = True,
                 optimistic: bool = False):
        """optimistic: the caller reads the training losses (train_losses_async) only after everything that depends
        on the training is queued, and repeats the pass on PlanHintMiss.  The launch is then queued with the
        capacities of the last plan read back for the same shapes (+ PLAN_HINT_MARGIN) instead of waiting for this
        one's -- the kernels compare them with the real plan on the device (hparams.owner_plan)."""
        K = self.n_shards = len(recs)
        tq = [("start", time.perf_counter())]                # host stamps of the constructor (diagnostics: ctor_ms)
        stamp = lambda name: tq.append((name, time.perf_counter()))
        if not 1 <= K <= _lib.URE_MAX_SHARDS:
            raise ValueError(f"1..{_lib.URE_MAX_SHARDS} shards per launch")
        if mode not in ("dense", "owner", "auto"):
            raise ValueError(f"mode {mode!r}")
        _need_cuda(*recs)
        L = _lib.lib()
        self.device = dev = recs[0].device
        self.epochs, self.lazy, self.decay = int(epochs), False, None
        self._recs, self._perms = list(recs), (list(perms) if perms is not None else [None] * K)
        self._rows_P, self._n_item, self._shard_ids = [int(r) for r in rows_P], int(n_item), [int(x) for x in shard_ids]
        self._perm_seed = int(perm_seed) & 0xFFFFFFFF
        ns = [int(r.shape[0]) for r in recs]
        self._ns = ns
        self.total_steps = max(-(-n // batch) for n in ns) * self.epochs
        self.hp = MFHParams(d=d, batch=batch, lr0=lr, lr_decay=lr_decay, lr_step=lr_step, weight_decay=weight_decay,
                            momentum=momentum, mode=_lib.MF_DENSE)
        self.owner_plan, self.launches_per_pass, self._shards = None, 0, None
        # warp groups of the DENSE schedule (greedy halves by interaction count)
        groups, load = [0] * K, [0, 0]
        if K >= 2:
            for j in sorted(range(K), key=lambda j: -ns[j]):
                g = 0 if load[0] <= load[1] else 1
                groups[j] = g
                load[g] += ns[j]
            w0 = int(round(32 * load[0] / max(1, load[0] + load[1])))
            self.warps_group0 = min(32 - 6, max(6, w0))
        else:
            self.warps_group0 = 32
        hs = (_lib.MFBatchShard * K)()
        for j in range(K):
            p = self._perms[j]
            if p is not None:
                assert p.dtype == torch.int32 and tuple(p.shape) == (self.epochs, ns[j]) and p.is_contiguous()
            hs[j].inter, hs[j].perm = recs[j].data_ptr(), (p.data_ptr() if p is not None else None)
            hs[j].n, hs[j].n_user, hs[j].shard_id, hs[j].group = ns[j], self._rows_P[j], self._shard_ids[j], groups[j]
        lay = _lib.MFBatchLayout()
        check(L.ure_mf_batch_layout(hs, K, n_item, d, batch, self.epochs, int(mode in ("owner", "auto")), OWNER_SCHED_BYTES,
                                    C.byref(lay)), "ure_mf_batch_layout")
        if mode == "owner" and not lay.owner:
            raise RuntimeError("owner mode does not fit this problem (row state beyond the SMs' shared memory)")
        self._lay = lay
        stamp("layout")
        self.arena = torch.empty(int(lay.total), dtype=torch.uint8, device=dev)
        base = self.arena.data_ptr()
        stage = _staging_bytes(176 * K + 64)
        stamp("alloc")
        self.table_ptr = base + int(lay.table)
        self.ws = self.arena[int(lay.ws):int(lay.ws) + int(L.ure_mf_train_workspace_bytes())]
        self.mode, self.optimistic, self.step = "dense", False, 0
        info = (C.c_int32 * 8)()
        force = OWNER_FORCE if OWNER_FORCE is not None else (-1, 0)
        sig = (K, d, batch, int(n_item), tuple(self._rows_P), self.epochs, perms is not None, bool(owner_cache),
               OWNER_FORCE, dev.index)

        def plan_with(vals):
            arr = (C.c_int32 * 4)(*[int(v) for v in vals])
            return L.ure_mf_batch_plan(arr, K, C.byref(self.hp), C.c_void_p(base), C.byref(lay),
                                       int(bool(owner_cache)), int(force[0]), int(force[1]), info)

        # optimistic: launch parameters from the remembered plan of these shapes, before anything is queued
        rc = 0
        hint = _PLAN_HINTS.get(sig) if (optimistic and lay.owner) else None
        if hint is not None:
            mr, ms, _, avail = hint
            for margin in (PLAN_HINT_MARGIN, 0.0):
                rc = plan_with((mr + int(mr * margin) + (2 if margin else 0), ms + int(ms * margin), lay.spe_cap, avail))
                if rc == 1:
                    break
            if rc == 1:
                self.optimistic, self.plan_sync_ms = True, 0.0
                self.hp.owner_plan = self.ws.data_ptr()
        with torch.cuda.device(dev):
            npass = 1
            while npass < 4 and (int(lay.max_rows) - 1) >> (8 * npass):
                npass += 1
            check(L.ure_mf_batch_setup(hs, K, n_item, C.byref(self.hp), self.epochs, self._perm_seed, C.c_void_p(base),
                                       C.byref(lay), C.c_void_p(stage.data_ptr()), 1 if self.optimistic else 0, _stream()),
                  "ure_mf_batch_setup")
            if lay.owner:
                # count + scan, radix passes, [inverse visiting orders], [plan]
                # one cooperative launch for batches of up to 8 M interactions (csrc/mf_batch.cu: flags & 8), unless
                # URE_SETUP_FUSED says otherwise
                try:
                    fused_env = int(os.environ.get("URE_SETUP_FUSED", "-1"))
                except ValueError:
                    fused_env = 0
                fused = fused_env > 0 or (fused_env < 0 and int(lay.n_total) <= (8 << 20))
                self.prepare_launches = (1 if fused else 2 + 3 * npass) + (1 if perms is not None else 0) + \
                    (0 if self.optimistic else 1)
                self.launches_per_pass += self.prepare_launches
            ev = torch.cuda.Event()
            ev.record()
        stamp("setup_queued")
        rows_w = int(lay.rows_total) + K * n_item

        def fill_weights():
            # weights: N(0, std) (reference utils.py:38-40), queued behind the set-up kernels -- and, on the optimistic
            # path, behind the schedule pre-pass, which does not read them (the host reaches that launch sooner)
            with torch.cuda.device(dev):
                self._W = self.arena[int(lay.W):int(lay.W) + rows_w * d * 4].view(torch.float32).view(rows_w, d)
                self._W.normal_(0.0, std, generator=generator() if callable(generator) else generator)

        if not self.optimistic:
            fill_weights()
        if lay.owner:
            if not self.optimistic:
                t0 = time.perf_counter()
                ev.synchronize()                             # the one wait of the set-up: upload + sorts + plan
                self.plan_sync_ms = (time.perf_counter() - t0) * 1e3
                plan = stage[176 * K:176 * K + 16].view(torch.int32)
                if len(_PLAN_HINTS) >= 256:                 # shapes come and go: the memory stays bounded
                    _PLAN_HINTS.clear()
                _PLAN_HINTS[sig] = tuple(int(v) for v in plan.tolist())
                rc = plan_with(plan.tolist())
            if rc < 0:
                check(rc, "ure_mf_batch_plan")
            self.owner_plan = dict(zip(("fits", "flags", "list_cap", "max_rows_per_cta", "max_slots_per_cta",
                                        "max_steps_per_epoch", "smem_need", "smem_avail"), list(info)))
            self.owner_plan["cached"] = bool(info[1] & 1) if info[1] >= 0 else False
            self.owner_plan["optimistic"] = self.optimistic
            self._plan_sig = sig
            if rc == 1:
                self.mode = "owner"
                self._sched_cover = (0, 0)
                self._spes = [-(-n // batch) for n in ns if n > 0]
                if self.optimistic:
                    self._schedule_window()              # the pre-pass is queued before anything else
                    stamp("schedule_queued")
                    fill_weights()
            elif mode == "owner":
                raise RuntimeError(f"owner mode does not fit this problem: {self.owner_plan}")
        _PINNED_BYTES.setdefault(stage.shape[0], []).append((stage, ev))
        stamp("end")
        self.ctor_ms = {b[0]: round((b[1] - a[1]) * 1e3, 4) for a, b in zip(tq[:-1], tq[1:])}

    # ---- what ShardBatch reads through self.table / self.shards
    @property
    def table(self):
        return _RawPtr(self.table_ptr)

    @property
    def shards(self):
        if self._shards is None:
            lay, d, K, E = self._lay, self.hp.d, len(self._recs), max(1, self.epochs)
            rows_w = int(lay.rows_total) + K * self._n_item
            Z = self.arena[int(lay.Z):int(lay.Z) + 2 * rows_w * d * 4].view(torch.float32).view(2, rows_w, d)
            sse = self.arena[int(lay.sse):int(lay.sse) + K * E * 8].view(torch.float64).view(K, E)
            out, o = [], 0
            for j in range(K):
                r, q = self._rows_P[j], int(lay.rows_total) + j * self._n_item
                out.append(ShardView(self._recs[j], self._W[o:o + r], self._W[q:q + self._n_item], Z[0, o:o + r],
                                     Z[0, q:q + self._n_item], Z[1, o:o + r], Z[1, q:q + self._n_item], sse[j],
                                     self._ns[j], self._shard_ids[j], self._perm_seed, self.epochs, self._perms[j]))
                o += r
            self._shards = out
        return self._shards

    def _upload_table(self):
        pass                                   # the descriptor table lives in the arena and never changes

    def _sse_matrix(self) -> torch.Tensor:
        lay, K, E = self._lay, self.n_shards, max(1, self.epochs)
        return self.arena[int(lay.sse):int(lay.sse) + K * E * 8].view(torch.float64).view(K, E)

    def _shard_sizes(self):
        return [max(1, n) for n in self._ns]

    def interactions_trained(self) -> int:
        return sum(self._ns) * self.epochs


class _RawPtr:
    """A bare device address with the one method _ptr() needs."""

    def __init__(self, p):
        self._p = int(p)

    def data_ptr(self):
        return self._p


def alloc_shard_batch(rows_P: Sequence[int], n_item: int, d: int, epochs: int, device, generator=None, std=1.0,
                      defer_init: bool = False):
    """One allocation for all shard models of a launch: N(0,std) tables (reference utils.py:38-40) plus the
    zero-filled momentum / gradient / loss scratch.  Returns per-shard (P, Q, scratch) views.
    defer_init=True returns (views, init): the memory is reserved, `init()` queues the fills -- pass it to
    ShardBatch(after_prepare=init) so the owner set-up's sorts are already running when the fills are launched."""
    K = len(rows_P)
    tot_p = int(sum(rows_P))
    W = torch.empty((tot_p + K * n_item, d), dtype=torch.float32, device=device)
    Z = torch.empty((2, tot_p + K * n_item, d), dtype=torch.float32, device=device)
    sse = torch.empty((K, max(1, epochs)), dtype=torch.float64, device=device)

    def init():
        W.normal_(0.0, std, generator=generator)
        Z.zero_()
        sse.zero_()

    if not defer_init:
        init()
    out, o = [], 0
    for j, r in enumerate(rows_P):
        qo = tot_p + j * n_item
        out.append((W[o:o + r], W[qo:qo + n_item],
                    (Z[0, o:o + r], Z[0, qo:qo + n_item], Z[1, o:o + r], Z[1, qo:qo + n_item], sse[j])))
        o += r
    return (out, init) if defer_init else out


# ------------------------------------------------------------------------------ evaluation
def ensemble_score(P_list, Q_list, inter, denom: Optional[float] = None, want_score: bool = True, sse=None):
    """(score fp32 [n] or None, sse fp64 [1]) for the K models (P_k, Q_k).  sse: a zeroed fp64 [1] to add into."""
    _need_cuda(inter, sse, *P_list, *Q_list)
    dev = inter.device
    K, d, n = len(P_list), P_list[0].shape[1], inter.shape[0]
    score = torch.empty(n, dtype=torch.float32, device=dev) if want_score else None
    if sse is None:
        sse = torch.zeros(1, dtype=torch.float64, device=dev)
    both = pointer_table(list(P_list) + list(Q_list), dev)      # one upload for both tables
    pt, qt = both[:K], both[K:]
    with torch.cuda.device(dev):
        check(_lib.lib().ure_ensemble_score(_ptr(pt), _ptr(qt), K, d, _ptr(inter), n,
                                            float(K if denom is None else denom), _ptr(score), _ptr(sse),
                                            _stream()), "ure_ensemble_score")
    return score, sse


def score_finalize(sum_t, inter, denom: float):
    _need_cuda(sum_t, inter)
    sse = torch.zeros(1, dtype=torch.float64, device=inter.device)
    score = torch.empty_like(sum_t)
    with torch.cuda.device(inter.device):
        check(_lib.lib().ure_score_finalize(_ptr(sum_t), _ptr(inter), inter.shape[0], float(denom), _ptr(score),
                                            _ptr(sse), _stream()), "ure_score_finalize")
    return score, sse


def user_segments(users: np.ndarray):
    """(order or None, seg int64 [n_seg+1]) grouping test rows by user id in order of first
    appearance with rows kept in file order (host dict of utils.py:151-161)."""
    users = np.asarray(users)
    n = len(users)
    if n == 0:
        return None, np.zeros(1, dtype=np.int64)
    change = np.flatnonzero(users[1:] != users[:-1]) + 1
    starts = np.concatenate([[0], change])
    if len(np.unique(users[starts])) == len(starts):        # every user is one contiguous run
        return None, np.concatenate([starts, [n]]).astype(np.int64)
    order = np.argsort(users, kind="stable")
    us = users[order]
    starts = np.concatenate([[0], np.flatnonzero(us[1:] != us[:-1]) + 1])
    return order.astype(np.int32), np.concatenate([starts, [n]]).astype(np.int64)


def user_segments_device(inter: torch.Tensor, n_user: int):
    """(order int32 [n], seg int64 [n_user + 1]) of the per-user test segments (utils.py:151-161), built ON the device
    without a host synchronisation by ure_user_segments: the owner set-up's stable radix sort on the user id (rows of
    a user stay in file order), CSR offsets by user id; users without test rows are empty segments (rank_metrics
    skips them).  The ranking metrics are sums over users, so the order of the segments does not matter."""
    _need_cuda(inter)
    n, dev = inter.shape[0], inter.device
    if n == 0 or n_user <= 0:
        return None, torch.full((max(0, n_user) + 1,), n, dtype=torch.int64, device=dev)
    L = _lib.lib()
    seg = torch.empty(n_user + 1, dtype=torch.int64, device=dev)
    order = torch.empty(n, dtype=torch.int32, device=dev)
    scratch = torch.empty(int(L.ure_user_segments_scratch_bytes(n, n_user)), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        check(L.ure_user_segments(_ptr(inter.contiguous()), n, n_user, _ptr(order), _ptr(seg), _ptr(scratch), _stream()),
              "ure_user_segments")
    return order, seg


def eval_jobs(jobs, d: int) -> torch.Tensor:
    """Many baseTest evaluations in one pair of launches (ure_eval_jobs).  jobs: list of (P_list, Q_list, inter, order
    or None, seg) -- device tensors; the ensemble mean divides by len(P_list).  Returns fp64 [n_jobs, 4] on the device:
    (sum of squared errors, sum NDCG@10, sum HR@10, users) per job, no synchronisation."""
    if not jobs:
        return torch.zeros((0, 4), dtype=torch.float64)
    dev = jobs[0][2].device
    ns = [int(j[2].shape[0]) for j in jobs]
    out = torch.zeros((len(jobs), 4), dtype=torch.float64, device=dev)
    score = torch.empty(max(1, sum(ns)), dtype=torch.float32, device=dev)
    ptrs = []
    for P_list, Q_list, *_ in jobs:
        assert len(P_list) == len(Q_list) >= 1
        ptrs += [t.data_ptr() for t in P_list] + [t.data_ptr() for t in Q_list]
    tab = upload_array(np.asarray(ptrs, dtype=np.int64), dev)
    arr = (_lib.EvalJob * len(jobs))()
    o = so = 0
    for x, (P_list, Q_list, inter, order, seg) in enumerate(jobs):
        _need_cuda(inter, order, seg, *P_list, *Q_list)
        m = len(P_list)
        a = arr[x]
        a.P, a.Q = tab.data_ptr() + 8 * o, tab.data_ptr() + 8 * (o + m)
        a.inter, a.order, a.seg = inter.data_ptr(), (order.data_ptr() if order is not None else None), seg.data_ptr()
        a.score, a.out = score.data_ptr() + 4 * so, out.data_ptr() + 32 * x
        a.n, a.n_seg, a.n_models, a.denom = ns[x], int(seg.shape[0]) - 1, m, float(m)
        o += 2 * m
        so += ns[x]
    d_jobs = upload_array(np.frombuffer(bytes(arr), dtype=np.uint8), dev)
    with torch.cuda.device(dev):
        check(_lib.lib().ure_eval_jobs(_ptr(d_jobs), len(jobs), int(d), max(ns), max(int(j[4].shape[0]) - 1 for j in jobs),
                                       _stream()), "ure_eval_jobs")
    out._keep = (tab, d_jobs, score, jobs)        # alive until the result has been read
    return out


def rank_metrics(inter, score, seg, order=None, out=None) -> torch.Tensor:
    """fp64 [3] = (sum ndcg, sum hr, #users).  out: a zeroed fp64 [3] to add into."""
    _need_cuda(inter, score, seg, order, out)
    if out is None:
        out = torch.zeros(3, dtype=torch.float64, device=inter.device)
    with torch.cuda.device(inter.device):
        check(_lib.lib().ure_rank_metrics(_ptr(inter), _ptr(score), _ptr(order), _ptr(seg), seg.shape[0] - 1,
                                          _ptr(out), _stream()), "ure_rank_metrics")
    return out


# ------------------------------------------------------------------------------ SISA bookkeeping
def route_deletions(owner: torch.Tensor, del_ids: torch.Tensor, n_shards: int) -> torch.Tensor:
    _need_cuda(owner, del_ids)
    flags = torch.zeros(n_shards, dtype=torch.int32, device=owner.device)
    with torch.cuda.device(owner.device):
        check(_lib.lib().ure_route_deletions(_ptr(owner), owner.shape[0], _ptr(del_ids), del_ids.shape[0],
                                             _ptr(flags), n_shards, _stream()), "ure_route_deletions")
    return flags


def merge_user_rows(P_list, owner, merged, row_of=None, retrain=None, zero_unowned=False) -> None:
    _need_cuda(owner, merged, row_of, retrain, *P_list)
    pt = pointer_table(P_list, merged.device)
    with torch.cuda.device(merged.device):
        check(_lib.lib().ure_merge_user_rows(_ptr(pt), _ptr(owner), _ptr(row_of), _ptr(retrain), _ptr(merged),
                                             merged.shape[0], merged.shape[1], int(zero_unowned), _stream()),
              "ure_merge_user_rows")


# ------------------------------------------------------------------------------ OT grouping
def kpad_for(k: int) -> int:
    """Columns a row of the cost matrix is stored with: 8 (32-byte rows: k <= 8 centroids are the common grouping,
    and a 64-byte row would be fetched from DRAM whole even if only half of it were read), else 16 .. 256."""
    for kp in (8, 16, 32, 64, 128, 256):
        if k <= kp:
            return kp
    raise ValueError("k > 256 centroids is not supported")


def cost_matrix(X, Cc, want_inertia=False, simt=False, out=None):
    """M [n,kpad] fp32 (columns >= k are +inf) and optionally the fp64 inertia scalar tensor.  out: an [n,kpad] fp32
    tensor to write into instead of a new one."""
    _need_cuda(X, Cc)
    n, d = X.shape
    k = Cc.shape[0]
    kp = kpad_for(k)
    if out is not None:
        assert out.shape == (n, kp) and out.dtype == torch.float32 and out.is_contiguous() and out.device == X.device
    M = torch.empty((n, kp), dtype=torch.float32, device=X.device) if out is None else out
    inertia = torch.zeros(1, dtype=torch.float64, device=X.device) if want_inertia else None
    fn = _lib.lib().ure_cost_matrix_simt if simt else _lib.lib().ure_cost_matrix
    with torch.cuda.device(X.device):
        check(fn(_ptr(X.contiguous()), n, d, _ptr(Cc.contiguous()), k, kp, _ptr(M), _ptr(inertia), _stream()),
              "ure_cost_matrix")
    return (M, inertia) if want_inertia else M


def sinkhorn(M, k, eps_schedule, g=None, tol: float = 0.0) -> torch.Tensor:
    """Single-GPU Sinkhorn; eps_schedule = [(eps, iters), ...], g = warm-start potentials (None: zeros),
    tol > 0 = early exit on the relative column-marginal error.  Returns g fp32 [k]."""
    _need_cuda(M, g)
    n, kp = M.shape
    g = torch.zeros(k, dtype=torch.float32, device=M.device) if g is None else g.clone()
    S = len(eps_schedule)
    eps = (C.c_float * S)(*[float(e) for e, _ in eps_schedule])
    its = (C.c_int32 * S)(*[int(i) for _, i in eps_schedule])
    ws = torch.zeros(int(_lib.lib().ure_sinkhorn_workspace_bytes()), dtype=torch.uint8, device=M.device)
    with torch.cuda.device(M.device):
        check(_lib.lib().ure_sinkhorn(_ptr(M), n, k, kp, _ptr(g), eps, its, S, float(tol), _ptr(ws), _stream()),
              "ure_sinkhorn")
    return g


_PEER_XCHG = {}      # (device index, world) -> (symmetric tensor, peer pointers, [call_base])
PEER_SINKHORN = True  # False: always the NCCL all-reduce loop (tests compare the two)


def _peer_exchange(dist, dev):
    """Symmetric (peer-mapped) exchange buffer of the fused multi-GPU Sinkhorn: allocated once per process through
    torch's symmetric-memory allocator, zero-filled, rendezvoused over the process group -> every rank's address."""
    key = (dev.index, dist.world)
    if key not in _PEER_XCHG:
        try:
            import torch.distributed._symmetric_memory as symm
            nbytes = int(_lib.lib().ure_sinkhorn_peer_xchg_bytes())
            t = symm.empty(nbytes // 8, dtype=torch.int64, device=dev)
            t.zero_()
            hdl = symm.rendezvous(t, dist.group if dist.group is not None else dist.td.group.WORLD)
            ptrs = [int(p) for p in hdl.buffer_ptrs]
            torch.cuda.synchronize(dev)
            dist.barrier()                                   # every buffer is zero before anybody's kernel runs
            _PEER_XCHG[key] = (t, hdl, ptrs, [1])
        except Exception as e:                               # no peer access (e.g. gloo / one GPU per node)
            _PEER_XCHG[key] = e
    got = _PEER_XCHG[key]
    return None if isinstance(got, Exception) else got


def sinkhorn_sharded(M, k, eps_schedule, dist, n_total, g=None, tol: float = 0.0) -> torch.Tensor:
    """Sinkhorn with the users (rows of M) sharded over the ranks of `dist`.  One rank: the single-GPU solver.
    Several GPUs with peer access: ONE persistent kernel per GPU that exchanges the k column sums through peer-mapped
    symmetric memory every iteration (ure_sinkhorn_peer).  Otherwise: column pass, all-reduce of the kpad column
    marginals, potential update per iteration.  Returns g fp32 [k], bit-identical on every rank."""
    if dist is None or dist.world == 1:
        return sinkhorn(M, k, eps_schedule, g=g, tol=tol)
    dev = M.device
    g = torch.zeros(k, dtype=torch.float32, device=dev) if g is None else g.clone()
    xchg = _peer_exchange(dist, dev) if (PEER_SINKHORN and M.is_cuda) else None
    if xchg is not None:
        _, _, ptrs, base = xchg
        S = len(eps_schedule)
        eps = (C.c_float * S)(*[float(e) for e, _ in eps_schedule])
        its = (C.c_int32 * S)(*[int(i) for _, i in eps_schedule])
        total = sum(int(i) for _, i in eps_schedule)
        ws = torch.zeros(int(_lib.lib().ure_sinkhorn_workspace_bytes()), dtype=torch.uint8, device=dev)
        arr = (C.c_uint64 * dist.world)(*ptrs)
        with torch.cuda.device(dev):
            check(_lib.lib().ure_sinkhorn_peer(_ptr(M), M.shape[0], float(n_total), k, M.shape[1], _ptr(g), eps, its, S,
                                               float(tol), arr, dist.rank, dist.world, base[0], _ptr(ws), _stream()),
                  "ure_sinkhorn_peer")
        base[0] += total + 2
        return g
    colsum = torch.zeros(M.shape[1], dtype=torch.float64, device=dev)
    for eps, iters in eps_schedule:
        for _ in range(int(iters)):
            sinkhorn_colsum(M, k, g, eps, n_total, colsum)
            dist.all_reduce(colsum)
            sinkhorn_update_g(g, colsum, k, eps)
    return g


def sinkhorn_colsum(M, k, g, eps, n_total, colsum) -> None:
    with torch.cuda.device(M.device):
        check(_lib.lib().ure_sinkhorn_colsum(_ptr(M), M.shape[0], k, M.shape[1], _ptr(g), float(eps),
                                             float(n_total), _ptr(colsum), _stream()), "ure_sinkhorn_colsum")


def sinkhorn_update_g(g, colsum, k, eps) -> None:
    with torch.cuda.device(g.device):
        check(_lib.lib().ure_sinkhorn_update_g(_ptr(g), _ptr(colsum), k, float(eps), _stream()),
              "ure_sinkhorn_update_g")


def sinkhorn_plan(M, k, g, eps, n_total=None) -> torch.Tensor:
    n, kp = M.shape
    plan = torch.empty((n, k), dtype=torch.float32, device=M.device)
    with torch.cuda.device(M.device):
        check(_lib.lib().ure_sinkhorn_plan(_ptr(M), n, k, kp, _ptr(g), float(eps),
                                           float(n if n_total is None else n_total), _ptr(plan), _stream()),
              "ure_sinkhorn_plan")
    return plan


def assign_plan(plan: torch.Tensor) -> torch.Tensor:
    """label = argmax_j plan[i,j], first maximum wins (utils.py:647)."""
    _need_cuda(plan)
    plan = plan.contiguous()
    n, k = plan.shape
    label = torch.empty(n, dtype=torch.int32, device=plan.device)
    fn = {torch.float64: _lib.lib().ure_assign_plan_f64, torch.float32: _lib.lib().ure_assign_plan_f32}[plan.dtype]
    with torch.cuda.device(plan.device):
        check(fn(_ptr(plan), n, k, k, _ptr(label), _stream()), "ure_assign_plan")
    return label


def assign_centroids(M, k, g, X=None):
    """(label int32 [n], sums fp64 [k,d] or None, counts int64 [k])."""
    n, kp = M.shape
    dev = M.device
    label = torch.empty(n, dtype=torch.int32, device=dev)
    cnt = torch.zeros(k, dtype=torch.int64, device=dev)
    d = 0 if X is None else X.shape[1]
    sums = None if X is None else torch.zeros((k, d), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        check(_lib.lib().ure_assign_centroids(_ptr(M), n, k, kp, _ptr(g), _ptr(X), d, _ptr(label), _ptr(sums),
                                              _ptr(cnt), _stream()), "ure_assign_centroids")
    return label, sums, cnt


def centroid_sums(X, label, k):
    """(sums fp64 [k,d], counts int64 [k]) of utils.py:648 for given labels (ure_centroid_sums)."""
    _need_cuda(X, label)
    n, d = X.shape
    sums = torch.zeros((k, d), dtype=torch.float64, device=X.device)
    cnt = torch.zeros(k, dtype=torch.int64, device=X.device)
    with torch.cuda.device(X.device):
        check(_lib.lib().ure_centroid_sums(_ptr(X), n, d, _ptr(label), k, _ptr(sums), _ptr(cnt), _stream()),
              "ure_centroid_sums")
    return sums, cnt


def balance_labels(M, k, label, cnt, max_aug: int = 1 << 14):
    """Balanced rounding in place (ure_balance_labels): `label` int32 [n] / `cnt` int64 [k] = an argmax assignment
    and its group sizes; afterwards every group holds floor(n/k)..ceil(n/k) users at minimum total cost.  Returns
    the int32 status tensor [3] = (augmentations, users still to move, gave-up flag) -- on the device, no sync."""
    _need_cuda(M, label, cnt)
    n, kp = M.shape
    assert label.dtype == torch.int32 and cnt.dtype == torch.int64 and label.shape[0] == n
    L = _lib.lib()
    ws = torch.empty(int(L.ure_balance_workspace_bytes(k)), dtype=torch.uint8, device=M.device)
    with torch.cuda.device(M.device):
        check(L.ure_balance_labels(_ptr(M), n, k, kp, _ptr(label), _ptr(cnt), int(max_aug), _ptr(ws), _stream()),
              "ure_balance_labels")
    return ws[128:140].view(torch.int32)


# ------------------------------------------------------------------------------ top-N recommendation
def _records_of(inters) -> torch.Tensor:
    """One int32 [n, 4] record tensor from one or several (device-to-device copies, no kernel)."""
    if isinstance(inters, torch.Tensor):
        return inters.contiguous()
    inters = [r for r in inters if r.shape[0] > 0] or list(inters[:1])
    if len(inters) == 1:
        return inters[0].contiguous()
    out = torch.empty((sum(r.shape[0] for r in inters), 4), dtype=torch.int32, device=inters[0].device)
    o = 0
    for r in inters:
        out[o:o + r.shape[0]].copy_(r, non_blocking=True)
        o += r.shape[0]
    return out


def seen_lists(inter, n_user: int, n_item: int):
    """(off int64 [n_user + 1], items int32 [n]): every user's training items in ascending order, built on the device by
    ure_seen_lists (the owner set-up's stable radix sort, by item and then by user).  `inter`: an int32 [n, 4] record
    tensor or a list of them (the shards' training sets); ids outside [0, n_user) / [0, n_item) raise ValueError."""
    inter = _records_of(inter)
    _need_cuda(inter)
    n, dev = inter.shape[0], inter.device
    if n > 0:           # the radix passes are sized by n_user / n_item: an id outside them would be mis-sorted silently
        u, i = inter[:, 0], inter[:, 1]
        if bool(((u < 0) | (u >= n_user) | (i < 0) | (i >= n_item)).any()):
            raise ValueError(f"seen_lists: user ids must lie in [0, {n_user}) and item ids in [0, {n_item})")
    L = _lib.lib()
    off = torch.empty(n_user + 1, dtype=torch.int64, device=dev)
    items = torch.empty(max(1, n), dtype=torch.int32, device=dev)
    scratch = torch.empty(int(L.ure_seen_lists_scratch_bytes(n, n_user)), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        check(L.ure_seen_lists(_ptr(inter), n, n_user, n_item, _ptr(off), _ptr(items), _ptr(scratch), _stream()),
              "ure_seen_lists")
    return off, items[:n]


def item_sum(Q_list) -> torch.Tensor:
    """S [n_item, d] = sum_k Q_k, summed in list order (ure_item_sum)."""
    _need_cuda(*Q_list)
    dev = Q_list[0].device
    n_item, d = Q_list[0].shape
    S = torch.empty((n_item, d), dtype=torch.float32, device=dev)
    qs = [q.contiguous() for q in Q_list]
    tab = pointer_table(qs, dev)
    with torch.cuda.device(dev):
        check(_lib.lib().ure_item_sum(_ptr(tab), len(qs), n_item, d, _ptr(S), _stream()), "ure_item_sum")
    S._keep = (tab, qs)
    return S


def recommend_topn(P, S, users, top_n: int, scale: float, seen=None):
    """(items int32 [m, top_n], scores fp32 [m, top_n]): for every id in `users` (int32 device tensor, any order,
    duplicates allowed) the top_n items of scale * P[u].S[i] over the whole catalogue, score descending, ties to the
    smaller item id, items of the user's seen list (``seen_lists``) excluded; short lists are padded with (-1, -inf).
    One tcgen05 launch (plus a merge launch when the item range is split over CTAs), no synchronisation."""
    _need_cuda(P, S, users)
    dev = P.device
    P, S = P.contiguous(), S.contiguous()
    users = users.to(device=dev, dtype=torch.int32).contiguous()
    n_user, d = P.shape
    n_item, m = S.shape[0], users.shape[0]
    L = _lib.lib()
    S_lo = torch.empty_like(S)
    items = torch.empty((m, top_n), dtype=torch.int32, device=dev)
    scores = torch.empty((m, top_n), dtype=torch.float32, device=dev)
    nb = int(L.ure_topn_scratch_bytes(m, n_item, d, top_n))
    scratch = torch.empty(nb, dtype=torch.uint8, device=dev) if nb > 0 else None
    off, seen_items = seen if seen is not None else (None, None)
    with torch.cuda.device(dev):
        check(L.ure_split_lo(_ptr(S), S.numel(), _ptr(S_lo), _stream()), "ure_split_lo")
        check(L.ure_topn(_ptr(P), n_user, _ptr(S), _ptr(S_lo), n_item, d, _ptr(users), m, _ptr(off), _ptr(seen_items),
                         int(top_n), float(scale), _ptr(items), _ptr(scores), _ptr(scratch), _stream()), "ure_topn")
    return items, scores


def topn_metrics(items, users, test_inter, n_user: int, seg=None, order=None) -> torch.Tensor:
    """fp64 [4] = (sum HR@N, sum Recall@N, sum NDCG@N, rows counted) of top-N lists against test records
    (ure_topn_metrics); the per-user test segments come from ``user_segments_device`` unless given."""
    _need_cuda(items, users, test_inter)
    dev = items.device
    out = torch.zeros(4, dtype=torch.float64, device=dev)
    if seg is None:
        order, seg = user_segments_device(test_inter, n_user)
    users = users.to(device=dev, dtype=torch.int32).contiguous()
    with torch.cuda.device(dev):
        check(_lib.lib().ure_topn_metrics(_ptr(items.contiguous()), _ptr(users), items.shape[0], items.shape[1],
                                          _ptr(test_inter.contiguous()), _ptr(order), _ptr(seg), n_user, _ptr(out),
                                          _stream()), "ure_topn_metrics")
    return out


# ------------------------------------------------------------------------------ learned combination of shard models
def combine_gram_entries(K: int) -> int:
    """Entries of one group's ure_combine_gram output: the upper triangle of the (K+1) x (K+1) Gram, the K+1 moments and
    the row count."""
    return (K + 1) * (K + 2) // 2 + (K + 1) + 1


def combine_gram(P, Q_list, inters) -> torch.Tensor:
    """fp64 [n_groups, combine_gram_entries(K)] on the device (ure_combine_gram): per record list of `inters` (int32
    [n, 4] each, one per group) the Gram of z = [x; 1] with x_k = P[u].Q_k[i], the moments sum z * r and the row count.
    Deterministic: the same bits on every call."""
    _need_cuda(P, *Q_list, *inters)
    dev = P.device
    K, d = len(Q_list), P.shape[1]
    E = combine_gram_entries(K)
    P = P.contiguous()
    qs = [q.contiguous() for q in Q_list]
    recs = [r.contiguous() for r in inters]
    out = torch.empty((len(recs), E), dtype=torch.float64, device=dev)
    if not recs:
        return out
    tab = upload_array(np.asarray([q.data_ptr() for q in qs] + [r.data_ptr() for r in recs] +
                                  [int(r.shape[0]) for r in recs], dtype=np.int64), dev)
    scratch = torch.empty(len(recs) * _lib.URE_COMBINE_GRAM_CTAS * E if K <= _lib.URE_COMBINE_MAX_MODELS else 1,
                          dtype=torch.float64, device=dev)
    G = len(recs)
    with torch.cuda.device(dev):
        check(_lib.lib().ure_combine_gram(_ptr(P), _ptr(tab), K, int(d), C.c_void_p(tab.data_ptr() + 8 * K),
                                          C.c_void_p(tab.data_ptr() + 8 * (K + G)), G, _ptr(out), _ptr(scratch),
                                          _stream()), "ure_combine_gram")
    out._keep = (tab, scratch, qs, recs)
    return out


def item_wsum(Q_list, w) -> torch.Tensor:
    """T [n_out, n_item, d] with T[o] = sum_k w[o, k] Q_k, in k order (ure_item_wsum); w: fp32 [n_out, K] on the device."""
    _need_cuda(w, *Q_list)
    dev = Q_list[0].device
    n_item, d = Q_list[0].shape
    K = len(Q_list)
    w = w.to(device=dev, dtype=torch.float32).contiguous()
    if w.dim() != 2 or w.shape[1] != K:
        raise ValueError(f"item_wsum: w must be [n_out, {K}]")
    T = torch.empty((w.shape[0], n_item, d), dtype=torch.float32, device=dev)
    qs = [q.contiguous() for q in Q_list]
    tab = pointer_table(qs, dev)
    with torch.cuda.device(dev):
        check(_lib.lib().ure_item_wsum(_ptr(tab), K, _ptr(w), int(w.shape[0]), n_item, d, _ptr(T), _stream()),
              "ure_item_wsum")
    T._keep = (tab, qs, w)
    return T


def group_score(P, T, b, owner, inter, sse=None):
    """(score fp32 [n], sse fp64 [1]) of ure_group_score: score = b[s] + P[u].T[s][i] with s = owner[u], or the last
    slot of T (the mean combination) for users in no group.  T: fp32 [n_slots, n_item, d]; b: fp32 [n_slots];
    owner: int32 [n_user].  sse: a zeroed fp64 [1] to add into."""
    _need_cuda(P, T, b, owner, inter, sse)
    dev = inter.device
    n = inter.shape[0]
    score = torch.empty(n, dtype=torch.float32, device=dev)
    if sse is None:
        sse = torch.zeros(1, dtype=torch.float64, device=dev)
    if T.dim() != 3 or b.shape != (T.shape[0],) or P.shape[1] != T.shape[2]:
        raise ValueError("group_score: T must be [n_slots, n_item, d] with b [n_slots] and P [n_user, d]")
    with torch.cuda.device(dev):
        check(_lib.lib().ure_group_score(_ptr(P.contiguous()), _ptr(T.contiguous()), int(T.shape[0]), int(T.shape[1]),
                                         int(T.shape[2]), _ptr(b.contiguous()), _ptr(owner.contiguous()),
                                         _ptr(inter.contiguous()), n, _ptr(score), _ptr(sse), _stream()),
              "ure_group_score")
    return score, sse
