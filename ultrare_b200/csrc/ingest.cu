// Data ingest on the device: the row filter and the shard split of readRating (reference read.py:36-68).
//
// The reference filters the ratings K times with np.in1d (one pass per group) minus the deleted users, and the
// B200 host mirror does one owner-map pass in NumPy; here the whole table is uploaded once and ONE stable
// partition by shard (a counting sort with the shard number as the only digit: per-CTA histograms, a scan, a
// rank-by-__match_any scatter) leaves every shard's packed records as one contiguous run in file order --
// exactly the rows, and the row order, of the reference's per-group arrays.
//
// Deleted ratings (interaction-level unlearning) go to the dropped bin in the same pass: with kDel the kernels take a
// per-user CSR of deleted items (del_off [n_map + 1], del_item ascending within a user, as ure_seen_lists builds it),
// and a row whose user has a non-empty list binary-searches its item there.  The rows of one user are usually
// adjacent in these files, so the offset reads of neighbouring lanes mostly hit the same lines.  Without lists
// (kDel = false) the kernels are the plain user filter.
#include "common.cuh"

namespace ure {
namespace {

constexpr int kPartThreads = 512;
constexpr int kPartWarps = kPartThreads / 32;
constexpr int kDropped = 255;             // bin of the rows that belong to no shard or to a deleted user

// Is `it` in the ascending list del_item[lo .. end)?
__device__ __forceinline__ bool listed(const int32_t* __restrict__ del_item, long long lo, long long end, int it) {
  long long hi = end;
  while (lo < hi) {                // lower bound of `it`
    const long long mid = (lo + hi) >> 1;
    if (del_item[mid] < it) lo = mid + 1; else hi = mid;
  }
  return lo < end && del_item[lo] == it;
}

// kDel: also drop the row when its item is in user u's deleted-item list del_item[del_off[u] .. del_off[u+1])
template <bool kDel>
__device__ __forceinline__ int shard_of(const double* __restrict__ cols, long long j, long long cs,
                                         const int32_t* __restrict__ owner, const unsigned char* __restrict__ deleted,
                                         int n_map, int n_shards, const long long* __restrict__ del_off,
                                         const int32_t* __restrict__ del_item) {
  const int u = (int)cols[j];      // callers pass j already multiplied by the row stride
  if (u < 0 || u >= n_map) return kDropped;
  if (deleted && deleted[u]) return kDropped;
  const int s = owner[u];
  if constexpr (kDel) {
    const long long lo = del_off[u], end = del_off[u + 1];
    if (lo < end && listed(del_item, lo, end, (int)cols[j + cs])) return kDropped;
  }
  return (s >= 0 && s < n_shards) ? s : kDropped;
}

// hist [grid.x][256]; the parameters after `hist` are read only by the kDel instantiation
template <bool kDel>
__global__ void __launch_bounds__(kPartThreads)
part_hist_kernel(const double* __restrict__ cols, long long n, long long rs, const int32_t* __restrict__ owner,
                 const unsigned char* __restrict__ deleted, int n_map, int n_shards, int* __restrict__ hist,
                 long long cs, const long long* __restrict__ del_off, const int32_t* __restrict__ del_item) {
  __shared__ int s_h[256];
  for (int x = threadIdx.x; x < 256; x += blockDim.x) s_h[x] = 0;
  __syncthreads();
  const long long tile = (n + gridDim.x - 1) / gridDim.x;
  const long long t0 = min(n, tile * blockIdx.x), t1 = min(n, t0 + tile);
  const int lane = threadIdx.x & 31;
  for (long long j0 = t0 + (threadIdx.x & ~31); j0 < t1; j0 += blockDim.x) {
    const long long j = j0 + lane;
    const bool in = j < t1;
    const int dg = in ? shard_of<kDel>(cols, j * rs, cs, owner, deleted, n_map, n_shards, del_off, del_item) : 0;
    const unsigned act = __ballot_sync(0xffffffffu, in);
    if (in) {
      const unsigned same = __match_any_sync(act, dg);
      if (lane == __ffs(same) - 1) atomicAdd(&s_h[dg], __popc(same));
    }
  }
  __syncthreads();
  for (int x = threadIdx.x; x < 256; x += blockDim.x) hist[(long long)blockIdx.x * 256 + x] = s_h[x];
}

// exclusive scan of hist in (bin, CTA) order, in place; the start of every bin's run -> shard_off[0 .. n_shards]
__global__ void __launch_bounds__(256)
part_scan_kernel(int* __restrict__ hist, int n_blocks, int n_shards, long long* __restrict__ shard_off) {
  __shared__ int s_tot[256];
  int* h = hist + threadIdx.x;
  int tot = 0;
  for (int b = 0; b < n_blocks; ++b) tot += h[b * 256];
  s_tot[threadIdx.x] = tot;
  __syncthreads();
  if (threadIdx.x < 32) {
    int loc[8], sum = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { loc[i] = sum; sum += s_tot[threadIdx.x * 8 + i]; }
    int inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int a = __shfl_up_sync(0xffffffffu, inc, o);
      if ((int)threadIdx.x >= o) inc += a;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) s_tot[threadIdx.x * 8 + i] = inc - sum + loc[i];
  }
  __syncthreads();
  int run = s_tot[threadIdx.x];
  if ((int)threadIdx.x <= n_shards) shard_off[threadIdx.x] = run;      // bins n_shards .. 254 are empty
  for (int b = 0; b < n_blocks; ++b) {
    const int t = h[b * 256];
    h[b * 256] = run;
    run += t;
  }
}

// the parameters after `out` are read only by the kDel instantiation
template <bool kDel>
__global__ void __launch_bounds__(kPartThreads)
part_scatter_kernel(const double* __restrict__ cols, long long n, long long rs, long long cs, double max_rating,
                    const int32_t* __restrict__ owner, const unsigned char* __restrict__ deleted, int n_map,
                    int n_shards, const int* __restrict__ hist, int4* __restrict__ out,
                    const long long* __restrict__ del_off, const int32_t* __restrict__ del_item) {
  __shared__ int s_wh[kPartWarps][256];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned lt = (1u << lane) - 1u;
  for (int x = threadIdx.x; x < kPartWarps * 256; x += blockDim.x) (&s_wh[0][0])[x] = 0;
  __syncthreads();
  const long long tile = (n + gridDim.x - 1) / gridDim.x;
  const long long t0 = min(n, tile * blockIdx.x), t1 = min(n, t0 + tile);
  const long long per = ((t1 - t0) + kPartWarps - 1) / kPartWarps;
  const long long w0 = min(t1, t0 + per * warp), w1 = min(t1, w0 + per);
  for (long long j0 = w0; j0 < w1; j0 += 32) {
    const long long j = j0 + lane;
    const bool in = j < w1;
    const int dg = in ? shard_of<kDel>(cols, j * rs, cs, owner, deleted, n_map, n_shards, del_off, del_item) : 0;
    const unsigned act = __ballot_sync(0xffffffffu, in);
    if (in) {
      const unsigned same = __match_any_sync(act, dg);
      if (lane == __ffs(same) - 1) s_wh[warp][dg] += __popc(same);
    }
    __syncwarp();
  }
  __syncthreads();
  if (threadIdx.x < 256) {
    int run = hist[(long long)blockIdx.x * 256 + threadIdx.x];
    for (int w = 0; w < kPartWarps; ++w) {
      const int t = s_wh[w][threadIdx.x];
      s_wh[w][threadIdx.x] = run;
      run += t;
    }
  }
  __syncthreads();
  for (long long j0 = w0; j0 < w1; j0 += 32) {
    const long long j = j0 + lane;
    const bool in = j < w1;
    const int dg = in ? shard_of<kDel>(cols, j * rs, cs, owner, deleted, n_map, n_shards, del_off, del_item) : 0;
    const unsigned act = __ballot_sync(0xffffffffu, in);
    if (in) {
      const unsigned same = __match_any_sync(act, dg);
      // read.py:64-68 + RatingData (read.py:111-113): float64 rating / max_rating, then float32
      const int4 rec = make_int4((int)cols[j * rs], (int)cols[j * rs + cs],
                                  __float_as_int((float)(cols[j * rs + 2 * cs] / max_rating)), 0);
      if (dg != kDropped) out[s_wh[warp][dg] + __popc(same & lt)] = rec;
      __syncwarp(act);
      if (lane == __ffs(same) - 1) s_wh[warp][dg] += __popc(same);
    }
    __syncwarp();
  }
}

__global__ void remap_users_kernel(const int4* __restrict__ in, long long n, const int32_t* __restrict__ row_of, int n_map,
                                   int4* __restrict__ out) {
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x) {
    int4 r = in[j];
    r.x = (r.x >= 0 && r.x < n_map) ? row_of[r.x] : -1;
    out[j] = r;
  }
}

}  // namespace
}  // namespace ure

extern "C" int ure_partition_blocks(void) { return 2 * ure::num_sms(); }

namespace ure {
namespace {
int partition(const double* d_cols, int64_t n, int64_t rs, int64_t cs, double max_rating, const int32_t* d_owner,
              const uint8_t* d_deleted, int32_t n_map, int n_shards, const int64_t* d_del_off, const int32_t* d_del_item,
              ure_inter_t* d_out, int32_t* d_hist, int64_t* d_shard_off, void* stream) {
  URE_REQUIRE(d_owner && d_hist && d_shard_off && ((d_cols && d_out) || n == 0), URE_EINVAL,
              "ure_partition_interactions: null argument");
  URE_REQUIRE(n_shards >= 1 && n_shards < kDropped, URE_EUNSUPPORTED,
              "ure_partition_interactions: n_shards=%d outside [1,%d]", n_shards, kDropped - 1);
  URE_REQUIRE(rs >= 1 && cs >= 1 && max_rating > 0.0 && n < (1ll << 31), URE_EINVAL,
              "ure_partition_interactions: bad strides / max_rating / n");
  URE_REQUIRE((d_del_off == nullptr) == (d_del_item == nullptr), URE_EINVAL,
              "ure_partition_interactions_del: d_del_off and d_del_item must both be set or both be NULL");
  auto st = static_cast<cudaStream_t>(stream);
  const int blocks = ure_partition_blocks();
  auto* off = reinterpret_cast<long long*>(d_shard_off);
  auto* out = reinterpret_cast<int4*>(d_out);
  auto* del_off = reinterpret_cast<const long long*>(d_del_off);
  if (del_off) {
    part_hist_kernel<true><<<blocks, kPartThreads, 0, st>>>(d_cols, n, rs, d_owner, d_deleted, n_map, n_shards, d_hist,
                                                            cs, del_off, d_del_item);
    part_scan_kernel<<<1, 256, 0, st>>>(d_hist, blocks, n_shards, off);
    part_scatter_kernel<true><<<blocks, kPartThreads, 0, st>>>(d_cols, n, rs, cs, max_rating, d_owner, d_deleted, n_map,
                                                               n_shards, d_hist, out, del_off, d_del_item);
  } else {
    part_hist_kernel<false><<<blocks, kPartThreads, 0, st>>>(d_cols, n, rs, d_owner, d_deleted, n_map, n_shards, d_hist,
                                                             cs, nullptr, nullptr);
    part_scan_kernel<<<1, 256, 0, st>>>(d_hist, blocks, n_shards, off);
    part_scatter_kernel<false><<<blocks, kPartThreads, 0, st>>>(d_cols, n, rs, cs, max_rating, d_owner, d_deleted, n_map,
                                                                n_shards, d_hist, out, nullptr, nullptr);
  }
  URE_CUDA(cudaGetLastError());
  return 0;
}
}  // namespace
}  // namespace ure

extern "C" int ure_partition_interactions(const double* d_cols, int64_t n, int64_t rs, int64_t cs, double max_rating,
                                          const int32_t* d_owner, const uint8_t* d_deleted, int32_t n_map,
                                          int n_shards, ure_inter_t* d_out, int32_t* d_hist, int64_t* d_shard_off,
                                          void* stream) {
  return ure::partition(d_cols, n, rs, cs, max_rating, d_owner, d_deleted, n_map, n_shards, nullptr, nullptr, d_out,
                        d_hist, d_shard_off, stream);
}

extern "C" int ure_partition_interactions_del(const double* d_cols, int64_t n, int64_t rs, int64_t cs,
                                              double max_rating, const int32_t* d_owner, const uint8_t* d_deleted,
                                              int32_t n_map, int n_shards, const int64_t* d_del_off,
                                              const int32_t* d_del_item, ure_inter_t* d_out, int32_t* d_hist,
                                              int64_t* d_shard_off, void* stream) {
  return ure::partition(d_cols, n, rs, cs, max_rating, d_owner, d_deleted, n_map, n_shards, d_del_off, d_del_item,
                        d_out, d_hist, d_shard_off, stream);
}

extern "C" int ure_remap_users(const ure_inter_t* d_in, int64_t n, const int32_t* d_row_of, int32_t n_map,
                               ure_inter_t* d_out, void* stream) {
  using namespace ure;
  URE_REQUIRE((d_in && d_out && d_row_of) || n == 0, URE_EINVAL, "ure_remap_users: null argument");
  if (n <= 0) return 0;
  const long long want = (n + 255) / 256, cap = 8ll * num_sms();
  const int blocks = (int)(want < cap ? want : cap);
  remap_users_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const int4*>(d_in), n, d_row_of,
                                                                          n_map, reinterpret_cast<int4*>(d_out));
  URE_CUDA(cudaGetLastError());
  return 0;
}
