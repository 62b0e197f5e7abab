import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from ultrare_b200 import kernels as kn
from ultrare_b200.method import utils as U
dev = torch.device("cuda:0")
rng = np.random.default_rng(7)
n, d, k = 6040, 16, 5
X = rng.standard_normal((n, d), dtype=np.float32)
Xd = torch.tensor(X, device=dev); Cd = torch.tensor(X[:k].copy(), device=dev)
def t(f, reps=20):
    f(); torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(reps): f()
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / reps * 1e3
M, inert = kn.cost_matrix(Xd, Cd, want_inertia=True)
scale = float(inert.item()) / n
sched = [(e * scale, i) for e, i in U.SINKHORN_SCHEDULE]
warm = [(e * scale, i) for e, i in U.SINKHORN_SCHEDULE[-U.SINKHORN_WARM_STAGES:]]
print("schedule", U.SINKHORN_SCHEDULE, "tol", U.SINKHORN_TOL, "warm stages", U.SINKHORN_WARM_STAGES)
print("cost_matrix ms", t(lambda: kn.cost_matrix(Xd, Cd, want_inertia=True)))
print("sinkhorn cold ms", t(lambda: kn.sinkhorn(M, k, sched, tol=U.SINKHORN_TOL)))
g = kn.sinkhorn(M, k, sched, tol=U.SINKHORN_TOL)
print("sinkhorn warm ms", t(lambda: kn.sinkhorn(M, k, warm, g=g, tol=U.SINKHORN_TOL)))
print("sinkhorn cold no tol ms", t(lambda: kn.sinkhorn(M, k, sched, tol=0.0)))
print("assign ms", t(lambda: kn.assign_centroids(M, k, g, Xd)))
np.random.seed(0); c0 = X[np.random.choice(n, k, replace=False)]
print("ot_cluster_device ms", t(lambda: U.ot_cluster_device(X, k, centroid0=c0, device=dev), reps=5))
# ---- balanced rounding makes the final labels independent of how far Sinkhorn converged (any potentials give the
# minimum-cost assignment for their own group sizes): what does a looser early-exit tolerance cost / save?
ref = None
for tol in (2e-5, 1e-4, 1e-3, 1e-2, 1e-1):
    ms = t(lambda: U.ot_cluster_device(X, k, centroid0=c0, device=dev, tol=tol), reps=5)
    inertia, label, cen, it = U.ot_cluster_device(X, k, centroid0=c0, device=dev, tol=tol)
    ref = label if ref is None else ref
    print(f"tol {tol:g}: {ms:.2f} ms, outer {it}, sizes {np.bincount(label, minlength=k).tolist()}, "
          f"agreement with tol 2e-5: {(label == ref).mean():.4f}, inertia {float(inertia):.3f}")
