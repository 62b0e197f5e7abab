import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from ultrare_b200 import kernels as kn, synth
dev = torch.device("cuda:0")
train, _ = synth.ml_like()
u, i, r = train
U, I, d, K = 6040, 3416, 16, 5
rs = np.random.RandomState(0)
groups = np.array_split(rs.permutation(U), K)
row_of = np.zeros(U, dtype=np.int64); owner = np.zeros(U, dtype=np.int64)
for g, ids in enumerate(groups):
    row_of[ids] = np.arange(len(ids)); owner[ids] = g
outs = []
for rep in range(4):
    shards = []
    gen = torch.Generator(device=dev).manual_seed(1)
    for g, ids in enumerate(groups):
        loc = owner[u] == g
        inter = kn.pack_interactions(row_of[u[loc]], i[loc], r[loc] / 5.0, dev)
        P = torch.empty((len(ids), d), device=dev).normal_(generator=gen)
        Q = torch.empty((I, d), device=dev).normal_(generator=gen)
        shards.append(kn.ShardState(inter, P, Q, 10, shard_id=g + 1, perm_seed=42))
    sb = kn.ShardBatch(shards, d, 30000, mode=sys.argv[1])
    sb.train(); torch.cuda.synchronize()
    outs.append((torch.cat([s.P.flatten() for s in shards] + [s.Q.flatten() for s in shards]).cpu().numpy(), np.concatenate(sb.train_losses())))
for rep in range(1, 4):
    print(sys.argv[1], "rep", rep, "max |dW| vs rep 0:", np.abs(outs[rep][0] - outs[0][0]).max(), "max |dloss|:", np.abs(outs[rep][1] - outs[0][1]).max())
print("final losses", outs[0][1][9::10])
