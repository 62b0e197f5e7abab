"""Benchmark of the sharded-retraining hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|c4|c5]
                    [--dump-outputs DIR]

--config c2 (default; BASELINE.json configs[1], the configuration the metric is quoted on): ml1m-shaped SISA,
    K=5 shards, retrain-after-delete with --delper 2 --deltype rand: route the 120 deleted users to their shards,
    retrain the affected shards from fresh weights for E=50 epochs (batch 30 000, SGD momentum 0.9, weight decay
    0.1), merge owner rows, ensemble-evaluate (RMSE / HR@10 / NDCG@10).  One "step" = one such pass.  Synthetic
    ML-1M-shaped data (ultrare_b200/synth.py); the K groups are a seeded balanced partition of the users -- the SAME
    one in both arms (OT grouping of the same users is timed beside it, `ot_grouping`).
    value = trained interactions / device time of the step, inputs resident in HBM (whole job, all ranks).
    e2e   = the same through the public API (ultrare_b200.method.sisa.Sisa.unlearn) from HOST numpy arrays in
            page-locked memory: H2D of this rank's shard and test interactions, record packing on the device, the
            pass, and D2H of the merged user table, the item tables and the metrics, wall clock between syncs.
    N > 1 : weak scaling -- every rank owns its own ml1m-shaped user population and 5 shards.
    The line also carries `check` (the step's RMSE against the CPU port run on the same groups, weights and
    visiting orders), `epoch_eval_modes` (what the drop-in's default per-epoch evaluation costs) and `c4_strong`
    (a slice of --config c4 at this N: the strong-scaling curve of north_star).
--config c3 | c4 : synthetic ml-20m shape (138 k x 27 k, 20 M, d=64, K=8) / 10 M x 1 M, 1 B, d=128, K=64: STRONG
    scaling of the fixed K (K/N shards per GPU, no training collective), one step = S global training steps.
--config c5 : Sinkhorn sweep n in {1 M, 10 M} x k in {8, 32, 128}, d=64, 100 iterations, users row-sharded over the
    ranks, column marginals reduced between the GPUs every iteration; float64 NumPy Sinkhorn timed beside it.
--impl reference : the oracle port of the reference's CPU path (oracle/mf.py, oracle/evalm.py, oracle/ot.py --
    vectorised PyTorch-CPU / NumPy on all host threads) on the same config; rank 0 alone runs it.
--dump-outputs DIR (--config c2, our arm): after the timed steps, what the last one returned to its caller (rank 0's
    view) is written as DIR/<name>.npy -- user_mat (the merged user table), item_mat (the item table of every shard
    on the rank), metrics (total RMSE / NDCG@10 / HR@10) and train_loss (every epoch of every retrained shard).  The inputs depend
    on the arguments only, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

A_MF = lambda d: 12 + 16 * d          # algorithmic bytes per trained interaction (SURVEY.md §8d)
K_SHARDS, D_EMB, BATCH, DEL_PER = 5, 16, 30000, 2
METRIC, UNIT = "mf_train_interactions_per_s (K-shard retrain-after-delete)", "interactions/s"
GROUP_SEED = 1

# name: (n_user, n_item, n_interactions, d, K, batch, shards per launch, global steps per bench step)
SHARD_CONFIGS = {
    "c3": (138_493, 26_744, 20_000_263, 64, 8, 30_000, 8, 84),
    "c4": (10_000_000, 1_000_000, 1_000_000_000, 128, 64, 30_000, 8, 100),
}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu, self.proc, self.path, self.skip = gpu_index, None, None, 0

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=open(self.path, "w"),
                                         stderr=subprocess.DEVNULL)
            t0 = time.time()                 # nvidia-smi needs ~0.1 s to come up: wait for its first line
            while time.time() - t0 < 2.0 and os.path.getsize(self.path) == 0:
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def mark(self):
        """Samples taken before this call (warm-up) are dropped by stop()."""
        try:
            self.skip = sum(1 for _ in open(self.path))
        except Exception:
            self.skip = 0

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in list(open(self.path))[self.skip:]:
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                sm.append(float(f[1])); mx.append(float(f[2]))
                for nm, v in zip(names, f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


# ----------------------------------------------------------------------------- c2 workload (both arms)
def host_workload(rank, epochs):
    """Host-side inputs of one rank: ml1m-shaped ratings, deletion set."""
    from ultrare_b200 import synth
    train, test = synth.ml_like(seed=synth.SEED + rank)
    n_user, n_item = synth.ML1M["n_user"], synth.ML1M["n_item"]
    rs = np.random.RandomState(0)
    n_del = int(DEL_PER / 100 * n_user)
    del_user = rs.choice(n_user, n_del, replace=False)                     # config.py:46-49 (+A1)
    return dict(train=train, test=test, n_user=n_user, n_item=n_item, del_user=del_user, epochs=epochs)


def bench_groups(n_user, k=K_SHARDS, seed=GROUP_SEED):
    """The step's user grouping in BOTH arms: a seeded balanced partition (exactly n/k users per group, as the
    reference's exact-EMD grouping gives -- SURVEY.md Appendix C).  The deletion set of config.py:46-49 (seed 0)
    spreads over all K groups of it, so all K shards retrain in both arms."""
    perm = np.random.RandomState(seed).permutation(n_user)
    return [sorted(int(u) for u in perm[i::k]) for i in range(k)]


def group_and_split(w, group_index, user_offset=0):
    """readRating(sort='a') semantics on in-memory columns, for learn (no deletion) and unlearn."""
    import pandas as pd
    from ultrare_b200.read import readRating
    tr = pd.DataFrame({0: w["train"][0], 1: w["train"][1], 2: w["train"][2]})
    te = pd.DataFrame({0: w["test"][0], 1: w["test"][1], 2: w["test"][2]})
    trr, idx = readRating(tr, w["n_user"], 5, [], [], K_SHARDS, group_index, "a")
    ter, _ = readRating(te, w["n_user"], 5, [], [], K_SHARDS, idx)
    trd, _ = readRating(tr, w["n_user"], 5, list(w["del_user"]), [], K_SHARDS, idx, "r")
    if user_offset:
        for arrs in (trr, ter, trd):
            for a in arrs:
                a[0] += user_offset
        idx = [[u + user_offset for u in g] for g in idx]
    return dict(learn_train=trr, unlearn_train=trd, test=ter, group_index=idx, del_user=w["del_user"] + user_offset)


def c2_config(world, n_inter_per_gpu, epochs, n_retrained, U1, I):
    """config of the c2 line -- the SAME dict in both arms (the driver compares them)."""
    return {"workload": "ml1m-shape SISA K=5/GPU retrain-after-delete (route + retrain affected shards + merge + "
                        "ensemble eval), delper=2 rand", "users_per_gpu": U1, "items": I,
            "train_interactions_per_gpu": int(n_inter_per_gpu), "epochs": epochs, "batch": BATCH, "d": D_EMB,
            "shards_per_gpu": K_SHARDS, "shards_retrained": int(n_retrained),
            "groups": f"seeded balanced partition (RandomState({GROUP_SEED})), same in both arms",
            "l2": "flushed between timed steps (256 MiB write)", "epoch_eval": "none",
            "parallelism": f"shards x{world} (no training collective)"}


class Param:
    def __init__(self, n_user, n_item, epochs, d=D_EMB):
        self.n_user, self.n_item, self.k, self.lam = n_user, n_item, d, 0.1
        self.seed, self.lr, self.lr_decay, self.momentum = 42, 0.001, 0.95, 0.9
        self.epochs, self.batch = epochs, BATCH


# ----------------------------------------------------------------------------- c2, our arm
def run_c2_ours(args):
    import torch
    from ultrare_b200 import dist as udist, kernels as kn
    from ultrare_b200.method.sisa import Sisa
    from ultrare_b200.method.utils import ot_cluster_device
    from ultrare_b200.read import RatingData, loadData

    d = udist.init_from_env()
    rank, world = d.rank, d.world
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    os.environ["ULTRARE_EPOCH_EVAL"] = "none"
    E = args.epochs

    w = host_workload(rank, E)
    U1, I = w["n_user"], w["n_item"]
    U = U1 * world
    # ---- OT grouping of this rank's users (timed separately; reported, not part of a step)
    rng = np.random.default_rng(7 + rank)
    emb = rng.standard_normal((U1, D_EMB), dtype=np.float32)
    np.random.seed(0)
    c0 = emb[np.random.choice(U1, K_SHARDS, replace=False)]
    ot_cluster_device(emb, K_SHARDS, centroid0=c0, device=dev)             # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, label, _, n_outer = ot_cluster_device(emb, K_SHARDS, centroid0=c0, device=dev)
    torch.cuda.synchronize()
    ot_ms = (time.perf_counter() - t0) * 1e3
    ot_sizes = np.bincount(label, minlength=K_SHARDS).tolist()
    sp = group_and_split(w, bench_groups(U1), user_offset=rank * U1)

    # global shard list: shard id = rank*5 + local (rank r owns ids with id // 5 == r)
    Kg = K_SHARDS * world
    mine_msg = dict(group_index=sp["group_index"], test=sp["test"], del_user=sp["del_user"])
    if world > 1:
        gathered = [None] * world
        d.td.all_gather_object(gathered, mine_msg)
    else:
        gathered = [mine_msg]
    group_index = [g for r in range(world) for g in gathered[r]["group_index"]]
    test_all = [t for r in range(world) for t in gathered[r]["test"]]
    del_user = np.concatenate([gathered[r]["del_user"] for r in range(world)])
    d.owner_of_shard = lambda s: s // K_SHARDS                              # block placement for this workload
    empty = np.zeros((3, 0))

    def loaders(key):
        tl = []
        for s in range(Kg):
            mine = s // K_SHARDS == rank
            tl.append(loadData(RatingData(sp[key][s % K_SHARDS] if mine else empty), BATCH, 1, True))
        return tl

    # the step's host inputs live in page-locked memory (the contract's "from pinned host memory"): the float64
    # [3, n] arrays readRating produced are copied there once, outside every timed region
    sp["unlearn_train"] = [kn.pinned_copy(a) for a in sp["unlearn_train"]]
    test_all = [kn.pinned_copy(t) for t in test_all]
    test_dlist = [loadData(RatingData(t), BATCH, 1, False) for t in test_all]
    test_np = kn.pinned_copy(np.hstack(test_all))
    test_data = loadData(RatingData(test_np), BATCH, 1, False)
    param = Param(U, I, E)

    def new_sisa(mode="none", cls=Sisa):
        s = cls(param, "mf", Kg, group_index)
        s.dist = d
        s.epoch_eval = mode
        return s

    # ---- learn once (setup, untimed): the models that exist before the deletion request
    learner = new_sisa()
    model_list = learner.learn(loaders("learn_train"), test_dlist, test_data, 0, "")
    torch.cuda.synchronize()

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    # ---- device-resident steps (value): loaders are reused so every record is already in HBM
    train_dl = loaders("unlearn_train")
    n_inter_local = sum(len(train_dl[s].dataset) for s in range(Kg) if s // K_SHARDS == rank)
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    step_ms = []
    total_steps = args.warmup + args.steps
    if rank == 0:
        sampler.start()
    for it in range(total_steps):
        if it == args.warmup and rank == 0:
            sampler.mark()
        flush.fill_(it & 0xFF)                                               # L2 flush between steps
        un = new_sisa()
        d.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        un.unlearn(model_list, train_dl, test_dlist, test_data, list(del_user), 0, "")
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if it >= args.warmup:
            step_ms.append(d.max_float(ms))
    if args.dump_outputs and rank == 0:
        # before anything reruns the batch: the kernel-alone repeats below retrain its tables in place
        dump_outputs(args.dump_outputs, un)
    if os.environ.get("URE_BENCH_TIMELINE") and rank == 0:
        # CUPTI timeline of one more device-resident step on rank 0 (every rank runs the step: collectives)
        from torch.profiler import ProfilerActivity, profile
        prof = profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA])
    else:
        prof = None
    if os.environ.get("URE_BENCH_TIMELINE"):
        flush.fill_(3)
        un = new_sisa()
        d.barrier()
        torch.cuda.synchronize()
        if prof is not None:
            prof.__enter__()
        un.unlearn(model_list, train_dl, test_dlist, test_data, list(del_user), 0, "")
        torch.cuda.synchronize()
        if prof is not None:
            prof.__exit__(None, None, None)
            evs = sorted([e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA],
                         key=lambda e: e.time_range.start)
            t0_, prev = evs[0].time_range.start, evs[0].time_range.start
            for e in evs:
                s_, en = e.time_range.start, e.time_range.end
                print(f"[timeline] {s_ - t0_:9.1f} {en - s_:9.1f} {s_ - prev:8.1f}  {e.name[:100]}", file=sys.stderr)
                prev = max(prev, en)
    n_retrained = len(un.retrain_gid)
    step_rmse = float(un.final_log["total_rmse"])
    sb = un._last_batch
    launches = int(getattr(sb, "launches_per_pass", 0) + un.timing.get("own_launches_outside_batch", 0)) * args.steps
    ms_per_step = float(np.mean(step_ms))
    inter_total = d.sum_int(n_inter_local) * E
    value = inter_total / (ms_per_step / 1e3)

    # ---- dominant kernel alone, on its launching stream (roofline)
    reps = max(3, args.steps)
    k_ms = []
    for _ in range(reps):
        sb.reset_for_rerun()
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sb.train()
        e1.record()
        torch.cuda.synchronize()
        k_ms.append(e0.elapsed_time(e1))
    kern_ms = float(np.median(k_ms))
    clocks = sampler.stop() if rank == 0 else None       # sampled over the timed steps + the kernel-alone repeats
    if os.environ.get("URE_BENCH_DEBUG"):
        print(f"[rank {rank}] last device-resident step: {un.timing}", file=sys.stderr)
    peak, peak_src = measured_peaks()
    alg_bytes = n_inter_local * E * A_MF(D_EMB)
    achieved = alg_bytes / (kern_ms / 1e3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "mf_train_traffic.json")
    kname = "mf_owner_kernel<16>" if sb.mode == "owner" else "mf_train_kernel<16>"
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(kname, {}).get("dram_bytes_per_launch")

    # ---- end to end from host buffers through the public API
    # uploaded per step: the float64 [3, n] arrays of this rank's shards and of the merged test set (the per-shard
    # test sets are only read by epoch_eval='final'/'faithful', not by this workload), the deletion list, the
    # shard descriptor table (N > 1: the test rows are sharded, a rank uploads the test sets of its own shards only)
    test_rows = test_np.shape[1] if world == 1 else sum(test_all[s].shape[1] for s in range(Kg) if s // K_SHARDS == rank)
    h2d = 24 * (sum(a.shape[1] for a in sp["unlearn_train"]) + test_rows) + 4 * len(del_user) + 176 * K_SHARDS
    e2e_ms = []
    d2h = 0
    # the loaders of an end-to-end step start their upload when they are BUILT (read.EAGER_UPLOAD_DEVICE: page-locked
    # arrays only), so the bytes travel while the step routes the deletions and lays out the batch
    from ultrare_b200 import read as ure_read
    ure_read.EAGER_UPLOAD_DEVICE = dev
    for it in range(args.warmup + args.steps):
        flush.fill_(it & 0xFF)
        d.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tl = loaders("unlearn_train")                                        # fresh: records are packed + uploaded
        tdl = [loadData(RatingData(t), BATCH, 1, False) for t in test_all]
        tdata = loadData(RatingData(test_np), BATCH, 1, False)
        t1 = time.perf_counter()
        un = new_sisa()
        t2 = time.perf_counter()
        ms_out = un.unlearn(model_list, tl, tdl, tdata, list(del_user), 0, "")
        t3 = time.perf_counter()
        # results to the host: the merged user table and this rank's item tables, one pinned transfer
        res_h = kn.download_many([ms_out[0].user_mat.weight.data] +
                                 [m.item_mat.weight.data for m in ms_out if getattr(m, "item_mat", None) is not None],
                                 copy=False)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) * 1e3
        e2e_parts = {"loaders_ms": (t1 - t0) * 1e3, "new_sisa_ms": (t2 - t1) * 1e3, "unlearn_ms": (t3 - t2) * 1e3,
                     "results_to_host_ms": dt - (t3 - t0) * 1e3}
        d2h = sum(x.size * 4 for x in res_h) + 24
        if it >= args.warmup:
            e2e_ms.append(d.max_float(dt))
    ure_read.EAGER_UPLOAD_DEVICE = None
    if os.environ.get("URE_BENCH_DEBUG"):
        print(f"[rank {rank}] e2e ms per step: {np.round(e2e_ms, 2).tolist()}; last: {e2e_parts} {un.timing}", file=sys.stderr)
    e2e_value = inter_total / (float(np.mean(e2e_ms)) / 1e3)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": c2_config(world, n_inter_local, E, n_retrained, U1, I),
        "retrain_after_delete_s": ms_per_step / 1e3,
        "interactions_per_s_per_gpu": value / world,
        "gpu_launches": launches,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": float(np.mean(e2e_ms)), "retrain_after_delete_s": float(np.mean(e2e_ms)) / 1e3},
        "roofline": {"bound": "hbm", "kernel": kname, "schedule": sb.mode, "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "kernel_ms": kern_ms, "algorithmic_bytes_per_launch": int(alg_bytes),
                     "share_of_step": kern_ms / ms_per_step,
                     "whole_step_frac": alg_bytes / (ms_per_step / 1e3) / 1e9 / peak,
                     "whole_step_frac_e2e": alg_bytes / (float(np.mean(e2e_ms)) / 1e3) / 1e9 / peak},
        "ot_grouping": {"ms": ot_ms, "n": U1, "k": K_SHARDS, "outer_iters": int(n_outer), "group_sizes": ot_sizes,
                        "balanced": ot_sizes == [U1 // K_SHARDS] * K_SHARDS},
    }
    if not args.no_extra:
        # ---- what the drop-in's other evaluation modes cost (Sisa.epoch_eval defaults to 'faithful')
        modes = {}
        for mode in ("final", "faithful"):
            if world > 1 and mode == "faithful":
                continue                                         # multi-GPU runs evaluate the last epoch only
            ts = []
            for rep in range(2):
                un_m = new_sisa(mode)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                un_m.unlearn(model_list, train_dl, test_dlist, test_data, list(del_user), 0, "")
                torch.cuda.synchronize()
                ts.append((time.perf_counter() - t0) * 1e3)
            modes[mode] = {"ms": float(min(ts)), "total_rmse": float(un_m.final_log["total_rmse"])}
        line["epoch_eval_modes"] = modes
        line["c4_strong"] = shard_training_leg("c4", d, dev, steps=100, reps=2)
        line["c3_strong"] = shard_training_leg("c3", d, dev, reps=2)
        # the C5 Sinkhorn sweep at this N (no CPU legs here: `--config c5` times the float64 NumPy Sinkhorn beside it)
        line["c5_sweep"] = [{k_: e[k_] for k_ in ("n", "k", "us_per_iter", "hbm_frac_per_gpu", "cost_matrix_ms", "cost_hbm_frac")}
                            for e in c5_sweep(d, dev, cpu=False)]
    if world > 1 and not args.no_extra:
        line["ot_sharded"] = ot_sharded_leg(d, dev)
    if rank == 0 and world == 1 and not args.no_cpu:
        # ---- the CPU port on the SAME groups, initial weights and visiting orders: the baseline and the checker
        class HostInitSisa(Sisa):
            init_on_device = False                               # N(0,1) tables from the host generator of scratch.py

        un_c = new_sisa("none", HostInitSisa)
        un_c.unlearn(model_list, train_dl, test_dlist, test_data, list(del_user), 0, "")
        gpu_rmse = float(un_c.final_log["total_rmse"])
        n_c, s_c, det = cpu_pass(sp, w, E, E, same_as_gpu=True)
        rel = abs(gpu_rmse - det["rmse"]) / det["rmse"]
        line["check"] = {"rmse_gpu": gpu_rmse, "rmse_cpu_port": det["rmse"], "rel_diff": rel, "tolerance": 1e-3,
                         "ok": bool(rel < 1e-3), "rmse_timed_step": step_rmse,
                         "what": "Sisa.unlearn with host-seeded N(0,1) weights vs oracle/mf.py + oracle/evalm.py on the "
                                 "same groups, weights and Feistel visiting orders, all epochs"}
        line["cpu_baseline"] = cpu_baseline_entry(n_c, s_c, det, E, E)
        line["cpu_baseline_as_shipped"] = as_shipped_entry(sp, w)
        if not line["check"]["ok"]:
            print(json.dumps(line))
            raise SystemExit(f"bench self-check failed: GPU RMSE {gpu_rmse} vs CPU port {det['rmse']}")
    if rank == 0:
        print(json.dumps(line))


def dump_outputs(out_dir, sisa):
    """What Sisa.unlearn gave its caller, as float32 / float64 .npy files under `out_dir` (about 1.5 MB at N=1)."""
    import torch
    mine = [m for m in sisa.model_list if getattr(m, "item_mat", None) is not None]
    arrays = {"user_mat": sisa.model_list[0].user_mat.weight.data,
              "item_mat": torch.stack([m.item_mat.weight.data for m in mine]),
              "metrics": np.array([sisa.final_log[k] for k in ("total_rmse", "total_ndcg", "total_hr")], dtype=np.float64),
              "train_loss": np.asarray(sisa.log["train_loss"], dtype=np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy() if torch.is_tensor(a) else a)


def ot_sharded_leg(d_, dev, n=2_000_000, k=8, dim=64, iters=100):
    """Row-sharded Sinkhorn over the ranks of this run (SURVEY.md §8e): the fused peer-memory kernel (one persistent
    launch per GPU, column sums exchanged through NVLink-mapped symmetric memory) against the per-iteration NCCL
    all-reduce loop on the same cost rows -- time per iteration of both and the largest difference of the potentials
    (driver-visible correctness evidence for the multi-GPU grouping path)."""
    import torch
    from ultrare_b200 import kernels as kn
    lo, hi = d_.row_block(n)
    X, cen = c5_inputs(hi - lo, k, dim, 100 + d_.rank)
    torch.manual_seed(5)
    C0 = cen + 0.5 * torch.randn((k, dim), device=dev)
    d_.td.broadcast(C0, 0)
    M, inert = kn.cost_matrix(X, C0, want_inertia=True)
    d_.all_reduce(inert)
    eps = 0.05 * float(inert.item()) / n
    out = {"n": n, "k": k, "d": dim, "iters": iters, "n_gpus": d_.world,
           "peer_memory": kn._peer_exchange(d_, dev) is not None}
    res = {}
    for name, flag in (("peer", True), ("nccl", False)):
        if name == "peer" and not out["peer_memory"]:
            continue
        kn.PEER_SINKHORN = flag
        ts = []
        for rep in range(3):
            d_.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g = kn.sinkhorn_sharded(M, k, [(eps, iters)], d_, n)
            e1.record()
            torch.cuda.synchronize()
            ts.append(d_.max_float(e0.elapsed_time(e1)))
        res[name] = g
        out[f"us_per_iter_{name}"] = min(ts) * 1e3 / iters
    kn.PEER_SINKHORN = True
    if "peer" in res:
        out["max_abs_diff_peer_vs_nccl"] = float((res["peer"] - res["nccl"]).abs().max().item())
        gs = [torch.empty_like(res["peer"]) for _ in range(d_.world)]
        d_.td.all_gather(gs, res["peer"])
        out["identical_on_all_ranks"] = bool(all(torch.equal(gs[0], x) for x in gs))
    peak, _ = measured_peaks()
    kp = M.shape[1]
    best = min(out.get("us_per_iter_peer", 1e30), out["us_per_iter_nccl"])
    out["hbm_frac_per_gpu"] = (4.0 * (hi - lo) * k + 8.0 * (hi - lo)) / (best * 1e-6) / 1e9 / peak
    return out


# ----------------------------------------------------------------------------- CPU arm (oracle port)
def cpu_pass(sp, w, epochs_sample, epochs_full, seed=42, same_as_gpu=False, user_offset=0):
    """The reference's CPU path for the c2 workload: the affected shards x `epochs_sample` epochs of baseTrain
    arithmetic + merge + ensemble baseTest; returns (interactions, seconds, detail).
    same_as_gpu: initial weights from scratch.model_generator(seed, id, 'cpu') and the keyed Feistel visiting orders
    -- what Sisa does with init_on_device=False -- so that the RMSE is comparable with the GPU step's."""
    import torch
    from oracle import evalm, mf as omf, sisa as osisa
    U, I = w["n_user"], w["n_item"]
    g = torch.Generator().manual_seed(seed)
    t_train = 0.0
    n_inter = 0
    Ps, Qs = [], []
    t0 = time.perf_counter()
    groups = [[u - user_offset for u in grp] for grp in sp["group_index"]] if user_offset else sp["group_index"]
    gid = osisa.route_deletions(groups, np.asarray(sp["del_user"]) - user_offset)
    t_route = time.perf_counter() - t0
    for s in sorted(gid):
        a = sp["unlearn_train"][s]
        u = torch.as_tensor((a[0] - user_offset).astype(np.int64)); i = torch.as_tensor(a[1].astype(np.int64))
        r = torch.as_tensor(a[2].astype(np.float32))
        if same_as_gpu:
            g = torch.Generator().manual_seed(int(seed) * 1000003 + (s + 1))      # scratch.model_generator
        P = torch.empty((U, D_EMB)).normal_(0.0, 1.0, generator=g); Q = torch.empty((I, D_EMB)).normal_(0.0, 1.0, generator=g)
        bP, bQ = torch.zeros_like(P), torch.zeros_like(Q)
        n = u.numel()
        step = 0
        for ep in range(epochs_sample):
            if same_as_gpu:
                perm = torch.as_tensor(omf.feistel_perm(n, omf.perm_key(seed, s + 1, ep)))
            else:
                perm = torch.randperm(n, generator=g)
            t0 = time.perf_counter()
            omf.mf_train_epoch_torch(P, Q, bP, bQ, u, i, r, perm, BATCH, omf.lr_at_epoch(1e-3, 0.95, ep), 0.1, 0.9, step)
            t_train += time.perf_counter() - t0
            step += -(-n // BATCH)
        n_inter += n * epochs_sample
        Ps.append(P.numpy()); Qs.append(Q.numpy())
    t0 = time.perf_counter()
    merged = osisa.merge_learn(Ps, [groups[s] for s in sorted(gid)])
    te = np.hstack(sp["test"])
    rmse, ndcg, hr, _ = evalm.base_test([merged] * len(Qs), Qs, (te[0] - user_offset).astype(np.int64),
                                        te[1].astype(np.int64), te[2].astype(np.float32))
    t_eval = time.perf_counter() - t0
    # the pass trains `epochs_full` epochs and evaluates once: prorate the one-off parts to the sample
    seconds = t_train + (t_route + t_eval) * epochs_sample / epochs_full
    return n_inter, seconds, dict(train_s=t_train, eval_s=t_eval, route_s=t_route, rmse=rmse, shards=len(gid))


def cpu_baseline_entry(n, s, det, epochs_sample, epochs_full):
    import torch
    full = epochs_sample == epochs_full
    return {"value": n / s, "unit": UNIT, "cores": torch.get_num_threads(), "host_cpus": os.cpu_count(), "kind": "port",
            "shards_retrained": det["shards"],
            "sample": (f"{det['shards']} shards x {epochs_sample} of {epochs_full} epochs of the vectorised PyTorch-CPU "
                       f"baseTrain port (oracle/mf.py) + ensemble baseTest port once"
                       + ("" if full else f" (prorated {epochs_sample}/{epochs_full})")
                       + f"; train {det['train_s']:.2f}s eval {det['eval_s']:.2f}s")}


def as_shipped_entry(sp, w, max_samples=60000):
    """BASELINE.md §3.1: the reference path as shipped (per-sample Dataset + DataLoader + autograd), bounded slice."""
    import torch
    from oracle import loader
    a = sp["unlearn_train"][0]
    workers = min(24, max(0, (os.cpu_count() or 1) - 1))                    # main.py:8 asks for 24
    try:
        n, s, loss = loader.as_shipped_epoch_slice(a[0], a[1], a[2], w["n_user"], w["n_item"], D_EMB, BATCH, workers,
                                                   max_samples=max_samples)
    except Exception as e:                                                    # e.g. no shared memory for workers
        workers = 0
        n, s, loss = loader.as_shipped_epoch_slice(a[0], a[1], a[2], w["n_user"], w["n_item"], D_EMB, BATCH, 0,
                                                   max_samples=max_samples)
    return {"value": n / s, "unit": UNIT, "cores": max(1, workers), "kind": "port (DataLoader path as shipped)",
            "extrapolated": True,
            "sample": f"first {n} interactions of shard 0, one pass through RatingData.__getitem__ + DataLoader("
                      f"batch={BATCH}, shuffle, num_workers={workers}) + autograd SGD (oracle/loader.py); a whole "
                      f"pass is this rate x {sum(x.shape[1] for x in sp['unlearn_train'])} interactions x epochs"}


def run_c2_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    torch.set_num_threads(os.cpu_count() or 1)            # torchrun exports OMP_NUM_THREADS=1
    world = max(1, args.gpus)
    E = args.epochs
    ep_s = args.cpu_epochs if args.cpu_epochs > 0 else (E if world == 1 else max(2, E // world))
    pops = []
    for r in range(world):                                # N > 1: the N populations of the weak-scaling workload
        w = host_workload(r, E)
        pops.append((w, group_and_split(w, bench_groups(w["n_user"]))))
    vals, secs, det = [], [], None
    for it in range(args.warmup + args.steps):
        n_tot, s_tot = 0, 0.0
        for w, sp in pops:
            n, s, det = cpu_pass(sp, w, ep_s, E, seed=42 + it)
            n_tot += n; s_tot += s
        if it >= args.warmup:
            vals.append(n_tot / s_tot); secs.append(s_tot * E / ep_s)
    v = float(np.mean(vals))
    w0, sp0 = pops[0]
    n_local = sum(a.shape[1] for a in sp0["unlearn_train"])
    base = cpu_baseline_entry(1, 1.0 / v, det, ep_s, E)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": float(np.mean(secs)) * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": c2_config(world, n_local, E, det["shards"], w0["n_user"], w0["n_item"]),
            "cpu_baseline": base, "epochs_sampled": ep_s, "populations": world,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ----------------------------------------------------------------------------- c3 / c4: strong scaling of fixed K
def shard_training_leg(name, d_, dev, steps=None, reps=3, mode="auto", e2e=False):
    """K shards of SHARD_CONFIGS[name] spread over the ranks (shard s on rank s mod N), trained `steps` global steps
    in rounds of at most R shards per launch; returns the leg's numbers (whole job, max over ranks)."""
    import torch
    from ultrare_b200 import kernels as kn, synth
    U, I, N, d, K, B, R, S = SHARD_CONFIGS[name]
    steps = S if steps is None else steps
    rank, world = d_.rank, d_.world
    mine = [s for s in range(K) if s % world == rank]
    rows_u, n_shard = U // K, N // K
    if mode == "auto" and (rows_u + I) <= 8 * B:
        # tables of the size of a batch: the owner schedule (rows resident in the SMs' shared memory) beats the dense
        # one whenever a launch's rows fit -- launch as many shards together as do (c3: ONE 22 MB shard at a time:
        # 2.5 G interactions/s against 2.0 for eight shards in one dense launch)
        from ultrare_b200 import _lib
        budget = int(_lib.lib().ure_mf_grid_size()) * (200 << 10)
        fit = max(1, budget // ((rows_u + I) * 8 * d))
        R = min(R, fit)
    rounds = [mine[x:x + R] for x in range(0, len(mine), R)]
    times, inter_local, mode_used, mem = [], 0, None, 0
    for rep in range(reps):
        t_ms, inter_local = 0.0, 0
        for grp in rounds:
            views = kn.alloc_shard_batch([rows_u] * len(grp), I, d, 1, dev,
                                         torch.Generator(device=dev).manual_seed(1 + rank), std=0.1)
            shards = []
            for j, s in enumerate(grp):
                rec = synth.device_interactions(rows_u, I, n_shard, dev, seed=synth.SEED + s)
                P, Q, scratch = views[j]
                shards.append(kn.ShardState(rec, P, Q, 1, shard_id=s + 1, perm_seed=42, scratch=scratch))
            big = (rows_u + I) > 8 * B                  # tables far larger than a batch: owner-computes in HBM
            sb = kn.ShardBatch(shards, d, B, mode=("runs" if big else "auto") if mode == "auto" else mode)
            mode_used = sb.mode
            n_steps = min(sb.total_steps, steps)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            sb.train(n_steps)
            sb.flush()
            e1.record()
            torch.cuda.synchronize()
            t_ms += e0.elapsed_time(e1)
            inter_local += sum(min(n_steps * B, s_.n) for s_ in shards)
            mem = max(mem, torch.cuda.max_memory_allocated() / 2**30)
            del sb, shards, views
            torch.cuda.empty_cache()
        d_.barrier()
        times.append(d_.max_float(t_ms))
    ms = float(np.min(times[1:] if len(times) > 1 else times))
    inter = d_.sum_int(inter_local)
    peak, _ = measured_peaks()
    alg = inter * A_MF(d)
    return {"workload": f"{name}: {U} users x {I} items, {N} interactions, d={d}, K={K} shards, batch {B}; {steps} global "
                        f"steps of every shard, {R} shard(s) per launch", "scaling": "strong", "n_gpus": world,
            "shards_per_gpu": len(mine), "schedule": mode_used, "interactions": int(inter), "ms": ms,
            "value": inter / ms * 1e3, "unit": UNIT, "interactions_per_s_per_gpu": inter / ms * 1e3 / world,
            "roofline_frac_per_gpu": alg / ms / 1e6 / world / peak, "mem_GB": mem, "launches_per_pass": len(rounds),
            "data": "synthetic, generated on the device (no host copy of 1 B interactions)"}


def run_shards_ours(args):
    import torch
    from ultrare_b200 import dist as udist
    d_ = udist.init_from_env()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    if d_.rank == 0:
        sampler.start()
    leg = shard_training_leg(args.config, d_, dev, reps=args.steps + 1)
    clocks = sampler.stop() if d_.rank == 0 else None
    U, I, N, d, K, B, R, S = SHARD_CONFIGS[args.config]
    peak, src = measured_peaks()
    line = {"metric": "mf_train_interactions_per_s (K-shard training, fixed K)", "value": leg["value"], "unit": UNIT,
            "n_gpus": d_.world, "steps": args.steps, "warmup": 1, "ms_per_step": leg["ms"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": leg["workload"], "parallelism": f"K/{d_.world} shards per GPU, no collective",
                       "l2": "inputs larger than L2 (c4) / flushed by the shard set-up between steps"},
            "interactions_per_s_per_gpu": leg["interactions_per_s_per_gpu"], "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": f"mf_train ({leg['schedule']})", "achieved": leg["roofline_frac_per_gpu"] * peak,
                         "peak": peak, "unit": "GB/s", "frac": leg["roofline_frac_per_gpu"], "traffic": None,
                         "peak_source": src},
            "e2e": None, "gpu_launches": args.steps * leg["launches_per_pass"], "detail": leg}
    if d_.rank == 0:
        print(json.dumps(line))


# ----------------------------------------------------------------------------- c5: Sinkhorn sweep
C5_POINTS = [(1_000_000, 8), (1_000_000, 32), (1_000_000, 128), (10_000_000, 8), (10_000_000, 32), (10_000_000, 128)]


def c5_inputs(n_local, k, d, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    cen = torch.randn((k, d), generator=g, device="cuda") * 2.0
    lab = torch.randint(0, k, (n_local,), generator=g, device="cuda")
    X = cen[lab] + torch.randn((n_local, d), generator=g, device="cuda")
    return X.contiguous(), cen.contiguous()


def run_c5_ours(args):
    import torch
    from ultrare_b200 import dist as udist
    d_ = udist.init_from_env()
    rank, world = d_.rank, d_.world
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    peak, src = measured_peaks()
    iters = 100
    out = c5_sweep(d_, dev, cpu=not args.no_cpu, iters=iters)
    if rank == 0:
        big = out[3]
        print(json.dumps({"metric": "sinkhorn_iterations_per_s (OT grouping sweep, c5)", "value": 1e6 / big["us_per_iter"],
                          "unit": "iterations/s", "n_gpus": world, "steps": iters, "warmup": 1,
                          "ms_per_step": big["us_per_iter"] / 1e3, "higher_is_better": True, "scaling": "strong",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": "c5: Sinkhorn sweep n in {1M,10M} x k in {8,32,128}, d=64, 100 "
                                                 "iterations at eps = 0.05 x mean nearest-centroid cost; headline = "
                                                 "n=10M, k=8", "parallelism": f"users row-sharded x{world}",
                                     "l2": "cost matrix larger than L2 at every point but n=1M, k=8 per 8 GPUs"},
                          "roofline": {"bound": "hbm", "kernel": "sinkhorn column pass", "frac": big["hbm_frac_per_gpu"],
                                       "achieved": big["hbm_frac_per_gpu"] * peak, "peak": peak, "unit": "GB/s",
                                       "traffic": None, "peak_source": src},
                          "e2e": None, "gpu_launches": iters, "sweep": out}))


def c5_sweep(d_, dev, cpu=False, iters=100, d=64, points=None):
    """The C5 points at this run's N: users row-sharded over the ranks, cost matrix + `iters` Sinkhorn iterations
    (single GPU: ure_sinkhorn; N > 1: the peer-memory kernel), whole-job time = max over ranks."""
    import torch
    from ultrare_b200 import kernels as kn
    rank, world = d_.rank, d_.world
    peak, _ = measured_peaks()
    out = []
    for n, k in (C5_POINTS if points is None else points):
        lo, hi = d_.row_block(n)
        X, cen = c5_inputs(hi - lo, k, d, 100 + rank)
        torch.manual_seed(5)
        C0 = cen + 0.5 * torch.randn((k, d), device=dev)
        if world > 1:
            d_.td.broadcast(C0, 0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        M, inert = kn.cost_matrix(X, C0, want_inertia=True)                  # warm-up; the inertia sets eps below
        torch.cuda.synchronize()
        e0.record()
        for _ in range(3):                    # back to back: the host's launch work hides behind the previous launch
            kn.cost_matrix(X, C0, want_inertia=True, out=M)
        e1.record()
        torch.cuda.synchronize()
        cost_ms = e0.elapsed_time(e1) / 3
        d_.all_reduce(inert)
        eps = 0.05 * float(inert.item()) / n
        runs = []
        for rep in range(2):
            g = torch.zeros(k, dtype=torch.float32, device=dev)
            d_.barrier()
            torch.cuda.synchronize()
            e0.record()
            g = kn.sinkhorn_sharded(M, k, [(eps, iters)], d_, n_total=n, g=g)
            e1.record()
            torch.cuda.synchronize()
            runs.append(d_.max_float(e0.elapsed_time(e1)))
        ms = min(runs)
        kp = M.shape[1]
        n_loc = hi - lo
        entry = {"n": n, "k": k, "d": d, "n_gpus": world, "iters": iters, "us_per_iter": ms * 1e3 / iters,
                 "hbm_frac_per_gpu": (4.0 * n_loc * k + 8.0 * n_loc) * iters / (ms / 1e3) / 1e9 / peak,
                 "algorithmic_bytes_per_iter_per_gpu": 4 * n_loc * k + 8 * n_loc, "kpad": kp,
                 "stored_bytes_per_iter_per_gpu": 4 * n_loc * kp + 8 * n_loc,
                 "cost_matrix_ms": cost_ms, "cost_GBps": (4.0 * n_loc * d + 4.0 * n_loc * kp) / (cost_ms / 1e3) / 1e9,
                 "cost_hbm_frac": (4.0 * n_loc * d + 4.0 * n_loc * kp) / (cost_ms / 1e3) / 1e9 / peak,
                 "cost_tflops": 2.0 * n_loc * kp * d / (cost_ms / 1e3) / 1e12}
        if rank == 0 and cpu:
            entry["cpu_float64_sinkhorn"] = c5_cpu_leg(X, C0, eps, iters, n if world == 1 else None)
        out.append(entry)
        del X, M
        torch.cuda.empty_cache()
    return out


def c5_cpu_leg(X, C0, eps, iters, n_full, budget_s=20.0):
    """float64 NumPy log-domain Sinkhorn (oracle/ot.py arithmetic) on the host at the same eps, as many of the
    `iters` iterations as fit the time budget -- no silent extrapolation: iterations done are reported."""
    import torch
    if n_full is None:
        return {"skipped": "multi-GPU run: the CPU leg is timed by the single-GPU run"}
    t0 = time.perf_counter()
    Xh = X.cpu().numpy().astype(np.float64)
    Ch = C0.cpu().numpy().astype(np.float64)
    M = (Xh * Xh).sum(1)[:, None] + (Ch * Ch).sum(1)[None, :] - 2.0 * Xh @ Ch.T          # chunk-free: [n,k] only
    t_cost = time.perf_counter() - t0
    n, k = M.shape
    g = np.zeros(k)
    loga, logb = -np.log(n), -np.log(k)
    done = 0
    t0 = time.perf_counter()
    while done < iters and time.perf_counter() - t0 < budget_s:
        T = (g[None, :] - M) / eps
        mx = T.max(axis=1, keepdims=True)
        lse = mx[:, 0] + np.log(np.exp(T - mx).sum(axis=1))
        col = np.exp(T + (loga - lse)[:, None]).sum(axis=0)
        g = g + eps * (logb - np.log(col))
        done += 1
    dt = time.perf_counter() - t0
    return {"iters_done": done, "of": iters, "seconds": dt, "us_per_iter": dt / max(1, done) * 1e6,
            "cost_matrix_s": t_cost, "status": "complete" if done == iters else f"CPU DNF @ {budget_s:.0f}s budget",
            "threads": torch.get_num_threads()}


def run_reference_other(args):
    """--impl reference for c3 / c4 / c5: the CPU port on a bounded sample of the same config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    from oracle import mf as omf
    if args.config == "c5":
        print(json.dumps({"impl": "reference", "unavailable": "c5: the CPU float64 Sinkhorn leg is timed inside the "
                          "single-GPU run of --config c5 (cpu_float64_sinkhorn per sweep point)"}))
        return
    U, I, N, d, K, B, R, S = SHARD_CONFIGS[args.config]
    rows_u, n = U // K, min(N // K, 2_000_000)
    rng = np.random.default_rng(0)
    u = torch.as_tensor((rng.random(n) ** 1.5 * rows_u).astype(np.int64).clip(max=rows_u - 1))
    i = torch.as_tensor((rng.random(n) ** 2.0 * I).astype(np.int64).clip(max=I - 1))
    r = torch.as_tensor(rng.integers(1, 6, n).astype(np.float32) / 5.0)
    g = torch.Generator().manual_seed(1)
    P = torch.empty((rows_u, d)).normal_(0, 0.1, generator=g); Q = torch.empty((I, d)).normal_(0, 0.1, generator=g)
    bP, bQ = torch.zeros_like(P), torch.zeros_like(Q)
    vals = []
    steps_cpu = 3
    for it in range(args.warmup + args.steps):
        perm = torch.randperm(n, generator=g)[:steps_cpu * B]
        t0 = time.perf_counter()
        omf.mf_train_epoch_torch(P, Q, bP, bQ, u, i, r, perm, B, 1e-3, 0.1, 0.9, 1)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            vals.append(steps_cpu * B / dt)
    v = float(np.mean(vals))
    print(json.dumps({"impl": "reference", "metric": "mf_train_interactions_per_s (K-shard training, fixed K)", "value": v,
                      "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": steps_cpu * B / v * 1e3, "higher_is_better": True, "scaling": "strong",
                      "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": f"{args.config}: one shard, {steps_cpu} steps of {B} (dense SGD sweep over "
                                             f"{rows_u}+{I} rows x d={d} every step, as the reference does)"},
                      "cpu_baseline": {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                                       "sample": f"{steps_cpu} steps of one {args.config} shard per bench step"},
                      "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "gpu_launches": 0}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=str, default="c2", choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--epochs", type=int, default=50)
    ap.add_argument("--cpu-epochs", type=int, default=0,
                    help="epochs per CPU sample of --impl reference (0 = all at N=1, epochs/N at N>1)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / check legs")
    ap.add_argument("--no-extra", action="store_true", help="skip the epoch_eval_modes / c4_strong legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (--config c2, --impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != "c2"):
        ap.error("--dump-outputs is implemented for --impl ours --config c2")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_c2_reference(args) if args.config == "c2" else run_reference_other(args)
    elif args.config == "c2":
        run_c2_ours(args)
    elif args.config == "c5":
        run_c5_ours(args)
    else:
        run_shards_ours(args)
    try:                                   # clean NCCL shutdown under torchrun (no warning after the JSON line)
        import torch.distributed as td
        if td.is_available() and td.is_initialized():
            td.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
