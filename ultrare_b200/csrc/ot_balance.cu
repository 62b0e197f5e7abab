// Balanced rounding of the Sinkhorn assignment (SURVEY.md H1 iv).
//
// The reference's transport plan is the exact EMD vertex (ot.emd, method/utils.py:641-644): for k | n every user
// carries a single entry 1/n and every group holds exactly n/k users, and label = argmax_j plan (utils.py:647) is
// the minimum-cost balanced assignment.  The argmax of the Sinkhorn plan, label_i = argmax_j (g_j - M_ij), is the
// minimum-cost assignment FOR ITS OWN group sizes (it minimises sum_i (M_i,label - g_label), and sum_i g_label is
// fixed by the sizes), which differ from n/k by a few users.  A min-cost flow that is optimal for its supplies
// stays optimal under successive shortest augmenting paths, so moving users from over-full to under-full groups
// along shortest paths of the k-node group graph
//     w(j -> l) = min over users i in group j of (M_il - M_ij)
// ends at the exact balanced optimum -- the EMD assignment whenever that optimum is unique.  Each augmentation moves
// one user per path edge; the edge weights are recomputed by one pass over M (n*k reads), Bellman-Ford runs on k
// nodes in shared memory.  The number of augmentations is the total surplus sum_j max(0, size_j - ceil(n/k)), a few
// dozen at ml1m size.  For k not dividing n every group ends with floor(n/k) or ceil(n/k) users.
#include "common.cuh"

namespace ure {
namespace {

constexpr int kBalThreads = 512;
constexpr unsigned long long kNone = 0xFFFFFFFFFFFFFFFFull;

struct BalWs {
  unsigned barrier;
  unsigned pad[31];
  int status[8];          // [0] augmentations applied, [1] users still to move, [2] 1 = gave up (cap / no path / cycle)
  // followed by W[2][k*k] packed edge minima (global buffers, multi-CTA launches only)
};

__device__ __forceinline__ unsigned ord_f32(float f) {       // order-preserving float -> unsigned
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float unord_f32(unsigned u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// One launch does every augmentation.  All CTAs keep identical copies of the group sizes and take identical
// decisions from the same reduced edge table; CTA 0 alone rewrites labels.
__global__ void __launch_bounds__(kBalThreads, 1)
balance_kernel(const float* __restrict__ M, long long n, int k, int kpad, int32_t* __restrict__ label,
               long long* __restrict__ cnt_io, int max_aug, BalWs* ws) {
  extern __shared__ __align__(16) unsigned char dyn[];
  unsigned long long* const s_W = reinterpret_cast<unsigned long long*>(dyn);              // [k*k] (ord(delta), user)
  unsigned long long* const s_dist = s_W + k * k;                                          // [k] (ord(dist), pred)
  int* const s_size = reinterpret_cast<int*>(s_dist + k);                                  // [k]
  int* const s_path = s_size + k;                                                          // [2*k] (user, new label)
  int* const s_par = s_path + 2 * k;                                                       // [k] predecessors (fallback)
  __shared__ int s_ctl[4];                 // [0] phase (0 done, 1 shed surplus, 2 fill deficit), [1] path edges, [2] changed
  const int tid = threadIdx.x;
  const bool multi = gridDim.x > 1;
  unsigned long long* const Wg = reinterpret_cast<unsigned long long*>(ws + 1);            // [2][k*k]
  const int lo = (int)(n / k), hi = (int)((n + k - 1) / k);
  for (int j = tid; j < k; j += kBalThreads) s_size[j] = (int)cnt_io[j];
  unsigned bar_target = 0;
  const long long per = (n + gridDim.x - 1) / gridDim.x;
  const long long r0 = min(n, per * blockIdx.x), r1 = min(n, r0 + per);
  int done = 0, gave_up = 0;
  __syncthreads();
  for (int it = 0;; ++it) {
    if (tid == 0) {
      int phase = 0;
      for (int j = 0; j < k; ++j) if (s_size[j] > hi) phase = 1;
      if (!phase) for (int j = 0; j < k; ++j) if (s_size[j] < lo) phase = 2;
      if (phase && it >= max_aug) { phase = 0; s_ctl[3] = 1; } else s_ctl[3] = 0;
      s_ctl[0] = phase;
    }
    for (int p = tid; p < k * k; p += kBalThreads) s_W[p] = kNone;
    if (multi && blockIdx.x == 0)          // the table of the NEXT iteration; this iteration's was reset one round ago
      for (int p = tid; p < k * k; p += kBalThreads) Wg[((it + 1) & 1) * k * k + p] = kNone;
    __syncthreads();
    const int phase = s_ctl[0];
    if (s_ctl[3]) gave_up = 1;
    if (!phase) break;
    // ---- edge weights: cheapest member of every group for every other group
    for (long long i = r0 + tid; i < r1; i += kBalThreads) {
      const int j = __ldcg(label + i);               // rewritten by CTA 0 between iterations: L2, not L1
      const float* row = M + i * kpad;
      const float mj = row[j];
      for (int l = 0; l < k; ++l) {
        if (l == j) continue;
        const unsigned long long pk = ((unsigned long long)ord_f32(row[l] - mj) << 32) | (unsigned)i;
        if (pk < s_W[j * k + l]) atomicMin(&s_W[j * k + l], pk);
      }
    }
    __syncthreads();
    if (multi) {
      unsigned long long* const W = Wg + (it & 1) * k * k;
      for (int p = tid; p < k * k; p += kBalThreads)
        if (s_W[p] != kNone) atomicMin(&W[p], s_W[p]);
      grid_barrier(&ws->barrier, bar_target);
      for (int p = tid; p < k * k; p += kBalThreads) s_W[p] = __ldcg(&W[p]);
      __syncthreads();
    }
    // ---- Bellman-Ford from every source at once (edges may be negative; a negative cycle only from fp32 rounding)
    for (int j = tid; j < k; j += kBalThreads) {
      const bool src = phase == 1 ? s_size[j] > hi : s_size[j] > lo;
      s_dist[j] = src ? (((unsigned long long)ord_f32(0.f) << 32) | 0xFFFFu) : kNone;
    }
    __syncthreads();
    int rounds = 0;
    for (;; ++rounds) {
      if (tid == 0) s_ctl[2] = 0;
      __syncthreads();
      for (int p = tid; p < k * k; p += kBalThreads) {
        const int j = p / k, l = p - j * k;
        const unsigned long long w = s_W[p], dj = s_dist[j];
        if (j == l || w == kNone || dj == kNone) continue;
        const float cand = unord_f32((unsigned)(dj >> 32)) + unord_f32((unsigned)(w >> 32));
        const unsigned long long pk = ((unsigned long long)ord_f32(cand) << 32) | (unsigned)j;
        // a shorter distance -- or the same distance through a lower group number, so that every CTA ends with the
        // same predecessors -- replaces the entry; only a shorter distance asks for another round
        const unsigned long long cur = s_dist[l];
        if (pk < cur) {
          atomicMin(&s_dist[l], pk);
          if ((pk >> 32) < (cur >> 32)) s_ctl[2] = 1;
        }
      }
      __syncthreads();
      const int changed = s_ctl[2];
      __syncthreads();
      if (!changed || rounds > k + 1) break;
    }
    // ---- cheapest sink, path back to its source, one user moved per edge
    if (tid == 0) {
      int sink = -1;
      unsigned best = 0xFFFFFFFFu;
      for (int j = 0; j < k; ++j) {
        const bool snk = phase == 1 ? s_size[j] < hi : s_size[j] < lo;
        const bool src = phase == 1 ? s_size[j] > hi : s_size[j] > lo;
        if (snk && !src && s_dist[j] != kNone && (unsigned)(s_dist[j] >> 32) < best) { best = (unsigned)(s_dist[j] >> 32); sink = j; }
      }
      int edges = 0;
      bool ok = sink >= 0 && rounds <= k + 1;
      if (ok) {
        int l = sink;
        while (true) {
          const int j = (int)(s_dist[l] & 0xFFFFu);
          if (j == 0xFFFF) break;                                   // reached a source
          if (edges >= k) { ok = false; break; }                    // the predecessors loop
          s_path[2 * edges] = (int)(s_W[j * k + l] & 0xFFFFFFFFu);
          s_path[2 * edges + 1] = l;
          ++edges;
          l = j;
        }
        if (ok) { s_size[l] -= 1; s_size[sink] += 1; }
      }
      // Exact and near ties -- a sparse rating row that shares no item with any centroid costs ||x||^2 + ||c_j||^2, and
      // thousands of users have the same cost differences up to the rounding of their row -- defeat the pass above in
      // three ways: the equal-distance rule closes the predecessors of a zero-weight cycle into a loop, fp32 distances
      // creep down around such a cycle until the round limit, and the rounding can make a swap of two tied users look an
      // ulp cheaper (a true negative cycle of the fp32 deltas).  Then this thread runs a strict Bellman-Ford from the
      // sources, the edge weights added in fp64 and only shorter distances replacing: a relaxation in round k + 1 means
      // a negative cycle, and one user moves along it (sizes unchanged, cost lower); otherwise the path to the cheapest
      // sink is a simple shortest path.  Where the pass above succeeds none of this runs.
      if (!ok && (sink >= 0 || rounds > k + 1)) {
        double* const d = reinterpret_cast<double*>(s_dist);      // s_dist is not read again in this round
        for (int j = 0; j < k; ++j) {
          const bool src = phase == 1 ? s_size[j] > hi : s_size[j] > lo;
          d[j] = src ? 0.0 : INFINITY;
          s_par[j] = -1;
        }
        int x = -1;
        for (int r = 0; r <= k; ++r) {
          x = -1;
          for (int j = 0; j < k; ++j) {
            if (d[j] == INFINITY) continue;
            for (int l = 0; l < k; ++l) {
              const unsigned long long w = s_W[j * k + l];
              if (l == j || w == kNone) continue;
              const double c = d[j] + (double)unord_f32((unsigned)(w >> 32));
              if (c < d[l]) { d[l] = c; s_par[l] = j; x = l; }
            }
          }
          if (x < 0) break;
        }
        if (x >= 0) {
          for (int t = 0; t < k; ++t) x = s_par[x];                 // onto the negative cycle
          int l = x;
          edges = 0;
          do {
            const int j = s_par[l];
            s_path[2 * edges] = (int)(s_W[j * k + l] & 0xFFFFFFFFu);
            s_path[2 * edges + 1] = l;
            ++edges;
            l = j;
          } while (l != x && edges <= k);
          ok = l == x;
        } else {
          int snk = -1;
          for (int j = 0; j < k; ++j) {
            const bool sj = phase == 1 ? s_size[j] < hi : s_size[j] < lo;
            const bool src = phase == 1 ? s_size[j] > hi : s_size[j] > lo;
            if (sj && !src && d[j] < INFINITY && (snk < 0 || d[j] < d[snk])) snk = j;
          }
          if (snk >= 0) {
            int l = snk;
            edges = 0;
            while (s_par[l] >= 0 && edges < k) {
              const int j = s_par[l];
              s_path[2 * edges] = (int)(s_W[j * k + l] & 0xFFFFFFFFu);
              s_path[2 * edges + 1] = l;
              ++edges;
              l = j;
            }
            if (s_par[l] < 0) { s_size[l] -= 1; s_size[snk] += 1; ok = true; }
          }
        }
      }
      s_ctl[1] = ok ? edges : -1;
    }
    __syncthreads();
    const int edges = s_ctl[1];
    if (edges < 0) { gave_up = 1; break; }
    if (blockIdx.x == 0 && tid < edges) label[s_path[2 * tid]] = s_path[2 * tid + 1];
    ++done;
    if (multi) grid_barrier(&ws->barrier, bar_target);            // the new labels are visible to every CTA
    else __syncthreads();
  }
  if (blockIdx.x == 0) {
    for (int j = tid; j < k; j += kBalThreads) cnt_io[j] = s_size[j];
    if (tid == 0) {
      int rest = 0;
      for (int j = 0; j < k; ++j) rest += max(0, s_size[j] - hi) + max(0, lo - s_size[j]);
      ws->status[0] = done; ws->status[1] = rest; ws->status[2] = gave_up;
    }
  }
}

}  // namespace
}  // namespace ure

extern "C" int64_t ure_balance_workspace_bytes(int k) {
  return (int64_t)sizeof(ure::BalWs) + 2ll * k * k * 8;
}

extern "C" int ure_balance_labels(const float* d_M, int64_t n, int k, int kpad, int32_t* d_label, int64_t* d_cnt,
                                  int max_aug, void* d_workspace, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_M && d_label && d_cnt && d_workspace, URE_EINVAL, "ure_balance_labels: null argument");
  URE_REQUIRE(n > 0 && k >= 1 && k <= kpad && k <= 128 && n < (1ll << 32), URE_EINVAL,
              "ure_balance_labels: bad shape n=%lld k=%d kpad=%d (k <= 128)", (long long)n, k, kpad);
  auto st = static_cast<cudaStream_t>(stream);
  auto* ws = static_cast<BalWs*>(d_workspace);
  URE_CUDA(cudaMemsetAsync(ws, 0, sizeof(BalWs), st));
  URE_CUDA(cudaMemsetAsync(ws + 1, 0xFF, 2ll * k * k * 8, st));
  if (k == 1) return 0;
  long long grid = (n + 8191) / 8192;
  if (grid > num_sms()) grid = num_sms();
  const size_t smem = (size_t)k * k * 8 + (size_t)k * 8 + (size_t)k * 4 + (size_t)k * 12 + 64;
  URE_CUDA(cudaFuncSetAttribute(balance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  long long nn = n;
  auto* cntp = reinterpret_cast<long long*>(d_cnt);
  void* args[] = {(void*)&d_M, (void*)&nn, (void*)&k, (void*)&kpad, (void*)&d_label, (void*)&cntp, (void*)&max_aug,
                  (void*)&ws};
  if (grid > 1) {
    URE_CUDA(cudaLaunchCooperativeKernel((void*)balance_kernel, dim3((unsigned)grid), dim3(kBalThreads), args, smem, st));
  } else {
    URE_CUDA(cudaLaunchKernel((void*)balance_kernel, dim3(1), dim3(kBalThreads), args, smem, st));
  }
  return 0;
}
