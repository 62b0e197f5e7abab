// 'rating-ot' grouping: the cost matrix and the centroid sums of the balanced OT clustering (reference utils.py:628-656)
// when the points are the users' sparse rating rows x_i (n_item columns, a few hundred nonzeros each) instead of a
// dense embedding.  Everything else of the outer loop -- Sinkhorn, arg-max labels, balanced rounding -- consumes the
// cost matrix these kernels write, unchanged.
//
//   cost:      M[i, j] = ||x_i||^2 - 2 x_i.c_j + ||c_j||^2 from the ratings ordered by user (CSR) and the centroid table
//              item-major (Ct [n_item, kpad]): every nonzero gathers one kpad-wide row of Ct.  About 2 kpad flops per
//              8 + 4 kpad bytes: a gather-bound kernel, no tensor cores.
//   centroids: per item the sums of the column's ratings by label, from the ratings ordered by item (CSC).
#include "common.cuh"

namespace ure {
namespace {

constexpr int kSpWarps = 8;                      // cost kernel: a CTA takes kSpWarps users, one warp per user
constexpr int kSpThreads = kSpWarps * 32;
constexpr int kSpLongRow = 1024;                 // a row with more nonzeros is taken by the whole CTA
constexpr int kCenWarps = 8;                     // centroid kernel: one warp per item
constexpr int kCountThreads = 256;

// Lane layout of a warp working on one row: CL = KP / 4 column lanes (lane c owns the centroid columns 4c .. 4c+3 and
// reads them with one 16-byte load) times NL = 32 / CL nonzero lanes.  The warp reads NL nonzeros per step, KP * 4
// bytes contiguous per nonzero (one 32-byte sector at k <= 8).  The dot products multiply the fp32 entries and add
// them in fp64: an fp32 dot product whose terms cancel misses the cost tolerance (combine.cu does the same).
// x_i is the summed row: the items of a row are ascending, so duplicate (user, item) entries are adjacent, and the first
// entry of a run stands for the run's fp32 sum (SciPy sums duplicates in the data type); the others add nothing.
template <int KP>
__device__ __forceinline__ void row_partial(const int32_t* __restrict__ item, const float* __restrict__ val,
                                            const float* __restrict__ Ct, long long rs, long long re, long long first,
                                            int stride, int c, double acc[4], double& nrm) {
  for (long long p = first; p < re; p += stride) {
    const int it = __ldg(item + p);
    if (p != rs && __ldg(item + p - 1) == it) continue;     // inside a run of duplicates: counted with its first entry
    float v = __ldg(val + p);
    for (long long r = p + 1; r < re && __ldg(item + r) == it; ++r) v += __ldg(val + r);
    const float4 q = __ldg(reinterpret_cast<const float4*>(Ct + (size_t)it * KP) + c);
    const double dv = (double)v;
    acc[0] = fma(dv, (double)q.x, acc[0]);
    acc[1] = fma(dv, (double)q.y, acc[1]);
    acc[2] = fma(dv, (double)q.z, acc[2]);
    acc[3] = fma(dv, (double)q.w, acc[3]);
    if (c == 0) nrm = fma(dv, dv, nrm);
  }
}

// Butterfly over the nonzero lanes (offsets CL .. 16): every lane ends with the sums of its column lane.
template <int CL>
__device__ __forceinline__ void reduce_nonzero_lanes(double acc[4]) {
#pragma unroll
  for (int o = CL; o < 32; o <<= 1)
#pragma unroll
    for (int t = 0; t < 4; ++t) acc[t] += __shfl_xor_sync(0xffffffffu, acc[t], o);
}

// The row's costs from the reduced sums (lanes 0 .. CL-1 store 16 bytes each) and its smallest real cost.
template <int KP>
__device__ __forceinline__ float row_store(const double acc[4], double nrm, const double* __restrict__ cnorm, int k,
                                           int c, bool store, float* __restrict__ Mrow) {
  constexpr int CL = KP / 4;
  float m[4];
  float rmin = INFINITY;
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const int j = 4 * c + t;
    m[t] = j < k ? (float)(nrm - 2.0 * acc[t] + __ldg(cnorm + j)) : INFINITY;
    rmin = fminf(rmin, m[t]);
  }
  if (store) reinterpret_cast<float4*>(Mrow)[c] = make_float4(m[0], m[1], m[2], m[3]);
#pragma unroll
  for (int o = 1; o < CL; o <<= 1) rmin = fminf(rmin, __shfl_xor_sync(0xffffffffu, rmin, o));
  return rmin;
}

// grid: ceil(n / kSpWarps) CTAs.  Warp w of CTA b takes user b * kSpWarps + w.  A row longer than kSpLongRow is left
// by its warp and taken afterwards by all kSpWarps warps of the CTA (the long-row path: ml1m rows run from 20 to
// ~2 300 nonzeros, C3 rows to several thousand, so one warp on such a row would keep its CTA waiting); their partial
// sums are added in warp order through shared memory.  part[b] = the CTA's sum of max(min_j M[i, j], 0) over its
// rows, added in warp order: sparse_inertia_kernel folds the parts in CTA order, so the inertia has the same bits on
// every call.  Four CTAs per SM (64 registers): left to itself, ptxas picks 32 registers and spills.
template <int KP>
__global__ void __launch_bounds__(kSpThreads, 4)
sparse_cost_kernel(const int64_t* __restrict__ off, const int32_t* __restrict__ item, const float* __restrict__ val,
                   long long n, const float* __restrict__ Ct, const double* __restrict__ cnorm, int k,
                   float* __restrict__ M, double* __restrict__ part) {
  constexpr int CL = KP / 4, NL = 32 / CL;
  __shared__ long long s_len[kSpWarps];
  __shared__ double s_acc[kSpWarps][KP];
  __shared__ double s_nrm[kSpWarps];
  __shared__ double s_inert[kSpWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = lane % CL, s = lane / CL;
  const long long u = (long long)blockIdx.x * kSpWarps + warp;
  long long rs = 0, re = 0;
  if (u < n) { rs = __ldg(off + u); re = __ldg(off + u + 1); }
  const bool lng = re - rs > kSpLongRow;
  if (lane == 0) s_len[warp] = u < n ? re - rs : 0;
  double inert = 0.0;
  if (u < n && !lng) {
    double acc[4] = {0.0, 0.0, 0.0, 0.0}, nrm = 0.0;
    row_partial<KP>(item, val, Ct, rs, re, rs + s, NL, c, acc, nrm);
    reduce_nonzero_lanes<CL>(acc);
    nrm = warp_sum(nrm);
    const float rmin = row_store<KP>(acc, nrm, cnorm, k, c, s == 0, M + (size_t)u * KP);
    inert = (double)fmaxf(rmin, 0.f);
  }
  __syncthreads();
  for (int w = 0; w < kSpWarps; ++w) {            // block-uniform: s_len is shared
    if (s_len[w] <= kSpLongRow) continue;
    const long long uw = (long long)blockIdx.x * kSpWarps + w;
    const long long ws = __ldg(off + uw), we = __ldg(off + uw + 1);
    double acc[4] = {0.0, 0.0, 0.0, 0.0}, nrm = 0.0;
    row_partial<KP>(item, val, Ct, ws, we, ws + warp * NL + s, kSpWarps * NL, c, acc, nrm);
    reduce_nonzero_lanes<CL>(acc);
    nrm = warp_sum(nrm);
    if (s == 0) {
#pragma unroll
      for (int t = 0; t < 4; ++t) s_acc[warp][4 * c + t] = acc[t];
    }
    if (lane == 0) s_nrm[warp] = nrm;
    __syncthreads();
    if (warp == 0) {
      double a[4] = {0.0, 0.0, 0.0, 0.0}, nr = 0.0;
      for (int x = 0; x < kSpWarps; ++x) {
#pragma unroll
        for (int t = 0; t < 4; ++t) a[t] += s_acc[x][4 * c + t];
        nr += s_nrm[x];
      }
      const float rmin = row_store<KP>(a, nr, cnorm, k, c, s == 0, M + (size_t)uw * KP);
      inert += (double)fmaxf(rmin, 0.f);
    }
    __syncthreads();
  }
  if (part) {
    if (lane == 0) s_inert[warp] = inert;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int x = 0; x < kSpWarps; ++x) t += s_inert[x];
      part[blockIdx.x] = t;
    }
  }
}

// *inertia += the parts, added in a fixed order (strided per thread, then a fixed tree).
__global__ void __launch_bounds__(256) sparse_inertia_kernel(const double* __restrict__ part, long long n_part,
                                                             double* __restrict__ inertia) {
  __shared__ double s[256];
  double t = 0.0;
  for (long long x = threadIdx.x; x < n_part; x += 256) t += part[x];
  s[threadIdx.x] = t;
  __syncthreads();
  for (int h = 128; h > 0; h >>= 1) {
    if ((int)threadIdx.x < h) s[threadIdx.x] += s[threadIdx.x + h];
    __syncthreads();
  }
  if (threadIdx.x == 0) *inertia += s[0];
}

// One warp per item.  The column's entries are read 32 at a time (user, rating, label[user]); then the warp walks them
// in column order, each broadcast to every lane, and lane l adds the rating to its accumulator of label l + 32 r.  So
// every (item, label) sum is added in the column's order, by one lane, in fp64: no floating-point atomics, the same bits
// on every call -- the next outer iteration's labels depend on these bits.  R = kpad / 32 accumulators per lane (1 for
// kpad <= 32).  sum [n_item, kpad]: every entry is written (0 for labels without a rating of the item and the pad).
// Duplicate (user, item) entries are adjacent (users ascending within a column): the first of a run carries the run's
// fp32 sum, the entry of SciPy's summed matrix, and the others carry nothing.
template <int KP>
__global__ void __launch_bounds__(kCenWarps * 32)
sparse_centroid_kernel(const int64_t* __restrict__ off, const int32_t* __restrict__ user, const float* __restrict__ val,
                       long long n_item, const int32_t* __restrict__ label, double* __restrict__ sum) {
  constexpr int R = KP < 32 ? 1 : KP / 32;
  const int lane = threadIdx.x & 31;
  const long long it = (long long)blockIdx.x * kCenWarps + (threadIdx.x >> 5);
  if (it >= n_item) return;                       // warp-uniform
  double acc[R];
#pragma unroll
  for (int r = 0; r < R; ++r) acc[r] = 0.0;
  const long long cs = __ldg(off + it), ce = __ldg(off + it + 1);
  for (long long p0 = cs; p0 < ce; p0 += 32) {
    const int cnt = ce - p0 < 32 ? (int)(ce - p0) : 32;
    int lab = -1;
    float v = 0.f;
    if (lane < cnt) {
      const long long p = p0 + lane;
      const int us = __ldg(user + p);
      if (p == cs || __ldg(user + p - 1) != us) {
        lab = __ldg(label + us);
        v = __ldg(val + p);
        for (long long r = p + 1; r < ce && __ldg(user + r) == us; ++r) v += __ldg(val + r);
      }
    }
    for (int x = 0; x < cnt; ++x) {
      const int lb = __shfl_sync(0xffffffffu, lab, x);
      const float vb = __shfl_sync(0xffffffffu, v, x);
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (lb == lane + 32 * r) acc[r] += (double)vb;
    }
  }
  double* out = sum + (size_t)it * KP;
#pragma unroll
  for (int r = 0; r < R; ++r)
    if (lane + 32 * r < KP) out[lane + 32 * r] = acc[r];
}

// cnt[j] += users with label j (integer atomics: the counts do not depend on the order).  Labels outside [0, k) are
// not counted.
__global__ void __launch_bounds__(kCountThreads) label_count_kernel(const int32_t* __restrict__ label, long long n, int k,
                                                                    unsigned long long* __restrict__ cnt) {
  __shared__ unsigned s_c[URE_SPARSE_OT_MAX_K];
  for (int j = threadIdx.x; j < k; j += blockDim.x) s_c[j] = 0u;
  __syncthreads();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int l = __ldg(label + i);
    if (l >= 0 && l < k) atomicAdd(&s_c[l], 1u);
  }
  __syncthreads();
  for (int j = threadIdx.x; j < k; j += blockDim.x)
    if (s_c[j]) atomicAdd(cnt + j, (unsigned long long)s_c[j]);
}

bool kpad_ok(int k, int kpad) {
  if (k < 1 || k > URE_SPARSE_OT_MAX_K) return false;
  int want = 8;
  while (want < k) want <<= 1;
  return kpad == want;
}

}  // namespace
}  // namespace ure

extern "C" int64_t ure_sparse_cost_scratch_bytes(int64_t n) {
  using namespace ure;
  return n > 0 ? (n + kSpWarps - 1) / kSpWarps * (int64_t)sizeof(double) : 0;
}

extern "C" int ure_sparse_cost(const int64_t* d_off, const int32_t* d_item, const float* d_val, int64_t n,
                               const float* d_Ct, const double* d_cnorm, int k, int kpad, float* d_M, double* d_inertia,
                               void* d_scratch, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_off && d_Ct && d_cnorm && d_M && n > 0 && (!d_inertia || d_scratch), URE_EINVAL,
              "ure_sparse_cost: bad argument (n=%lld)", (long long)n);
  URE_REQUIRE(kpad_ok(k, kpad), URE_EUNSUPPORTED, "ure_sparse_cost: k=%d kpad=%d (need 1 <= k <= %d, kpad = 8 .. 128 "
              "the smallest power of two >= max(k, 8))", k, kpad, URE_SPARSE_OT_MAX_K);
  auto st = static_cast<cudaStream_t>(stream);
  const long long blocks = (n + kSpWarps - 1) / kSpWarps;
  URE_REQUIRE(blocks < (1ll << 31), URE_EUNSUPPORTED, "ure_sparse_cost: n=%lld too large", (long long)n);
  double* part = d_inertia ? static_cast<double*>(d_scratch) : nullptr;
  switch (kpad) {
    case 8: sparse_cost_kernel<8><<<(unsigned)blocks, kSpThreads, 0, st>>>(d_off, d_item, d_val, n, d_Ct, d_cnorm, k, d_M, part); break;
    case 16: sparse_cost_kernel<16><<<(unsigned)blocks, kSpThreads, 0, st>>>(d_off, d_item, d_val, n, d_Ct, d_cnorm, k, d_M, part); break;
    case 32: sparse_cost_kernel<32><<<(unsigned)blocks, kSpThreads, 0, st>>>(d_off, d_item, d_val, n, d_Ct, d_cnorm, k, d_M, part); break;
    case 64: sparse_cost_kernel<64><<<(unsigned)blocks, kSpThreads, 0, st>>>(d_off, d_item, d_val, n, d_Ct, d_cnorm, k, d_M, part); break;
    default: sparse_cost_kernel<128><<<(unsigned)blocks, kSpThreads, 0, st>>>(d_off, d_item, d_val, n, d_Ct, d_cnorm, k, d_M, part); break;
  }
  URE_CUDA(cudaGetLastError());
  if (d_inertia) {
    sparse_inertia_kernel<<<1, 256, 0, st>>>(part, blocks, d_inertia);
    URE_CUDA(cudaGetLastError());
  }
  return 0;
}

extern "C" int ure_sparse_centroid_sums(const int64_t* d_off, const int32_t* d_user, const float* d_val, int64_t n_item,
                                        const int32_t* d_label, int64_t n_user, int k, int kpad, double* d_sum,
                                        int64_t* d_cnt, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_off && d_label && d_sum && d_cnt && n_item > 0 && n_user > 0, URE_EINVAL,
              "ure_sparse_centroid_sums: bad argument (n_item=%lld, n_user=%lld)", (long long)n_item, (long long)n_user);
  URE_REQUIRE(kpad_ok(k, kpad), URE_EUNSUPPORTED, "ure_sparse_centroid_sums: k=%d kpad=%d (need 1 <= k <= %d, kpad = "
              "8 .. 128 the smallest power of two >= max(k, 8))", k, kpad, URE_SPARSE_OT_MAX_K);
  auto st = static_cast<cudaStream_t>(stream);
  const long long blocks = (n_item + kCenWarps - 1) / kCenWarps;
  URE_REQUIRE(blocks < (1ll << 31), URE_EUNSUPPORTED, "ure_sparse_centroid_sums: n_item=%lld too large", (long long)n_item);
  switch (kpad) {
    case 8: sparse_centroid_kernel<8><<<(unsigned)blocks, kCenWarps * 32, 0, st>>>(d_off, d_user, d_val, n_item, d_label, d_sum); break;
    case 16: sparse_centroid_kernel<16><<<(unsigned)blocks, kCenWarps * 32, 0, st>>>(d_off, d_user, d_val, n_item, d_label, d_sum); break;
    case 32: sparse_centroid_kernel<32><<<(unsigned)blocks, kCenWarps * 32, 0, st>>>(d_off, d_user, d_val, n_item, d_label, d_sum); break;
    case 64: sparse_centroid_kernel<64><<<(unsigned)blocks, kCenWarps * 32, 0, st>>>(d_off, d_user, d_val, n_item, d_label, d_sum); break;
    default: sparse_centroid_kernel<128><<<(unsigned)blocks, kCenWarps * 32, 0, st>>>(d_off, d_user, d_val, n_item, d_label, d_sum); break;
  }
  URE_CUDA(cudaGetLastError());
  URE_CUDA(cudaMemsetAsync(d_cnt, 0, (size_t)k * sizeof(int64_t), st));
  long long cb = (n_user + kCountThreads - 1) / kCountThreads;
  if (cb > 2 * num_sms()) cb = 2 * num_sms();
  label_count_kernel<<<(unsigned)cb, kCountThreads, 0, st>>>(d_label, n_user, k,
                                                           reinterpret_cast<unsigned long long*>(d_cnt));
  URE_CUDA(cudaGetLastError());
  return 0;
}
