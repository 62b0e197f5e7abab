// Learned combination of the SISA shard models (UltraRE's combination estimator): per owner group g a ridge fit
//   s(u, i) = b_g + sum_k w_gk x_k,   x_k = P[u].Q_k[i]   (P the merged user table, Q_k the shard item tables)
// which is b_g + P[u].T_g[i] with T_g = sum_k w_gk Q_k.  Here: the Gram of the features over a group's training rows
// (the (K+1) x (K+1) solve runs on the host in float64), the weighted item tables T_g, and the per-group test scores.
#include "common.cuh"

namespace ure {
namespace {

constexpr int kGramThreads = 256;
constexpr int kGramTile = 128;                 // records staged in shared memory per round (a multiple of 256 / (D/4))
constexpr int kGramStride = URE_COMBINE_MAX_MODELS + 3;   // z row: x_0 .. x_{K-1}, 1, r (odd stride: fewer bank conflicts)
constexpr int kGramMaxPer = 9;                 // entries per thread: ceil(gram_entries(64) / 256)

// Entries of one group's output, in order: the upper triangle of sum [x;1][x;1]^T row by row ((K+1)(K+2)/2 values),
// then sum [x;1] * r (K+1 values), then the row count.  Entry e is the sum over rows of z_a * z_b with z = [x; 1; r].
__host__ __device__ constexpr int gram_entries(int K) { return (K + 1) * (K + 2) / 2 + (K + 1) + 1; }

__device__ __forceinline__ void gram_pair(int e, int K, int& a, int& b) {
  const int U = (K + 1) * (K + 2) / 2;
  if (e < U) {
    int row = K + 1, r = 0;
    while (e >= row) { e -= row; --row; ++r; }
    a = r; b = r + e;
  } else if (e < U + K + 1) {
    a = e - U; b = K + 1;
  } else {
    a = K; b = K;                              // 1 * 1: the row count
  }
}

// grid (URE_COMBINE_GRAM_CTAS, n_groups).  CTA c of group g takes the tiles c, c + CTAS, ... of the group's records, so
// which rows a CTA adds, and in which order, depends on the row count only.  Per tile: the features of kGramTile
// records into shared memory (D/4 lanes per record, the P row once, one 16-byte load per lane and model; the same dot
// product for every k, with the products of the fp32 entries formed and summed in fp64 -- an fp32 dot product loses
// most of its digits when the terms cancel, and a group of a few rows would carry that error into its Gram), then
// every thread adds z_a * z_b in fp64 for its entries.  With few entries the threads split into R copies that take
// every R-th record; the copies are folded in copy order, the CTA's partials go to `part`, and gram_fold_kernel adds
// them in CTA order: no floating-point atomics, the same bits on every call.
template <int D>
__global__ void __launch_bounds__(kGramThreads)
combine_gram_kernel(const float* __restrict__ P, const float* const* __restrict__ Q, int K,
                    const ure_inter_t* const* __restrict__ inter, const int64_t* __restrict__ n_rows,
                    double* __restrict__ part) {
  constexpr int G = D / 4;
  constexpr int RPP = kGramThreads / G;        // records per pass of the feature phase
  static_assert(kGramTile % RPP == 0, "uniform trip count of the feature phase");
  extern __shared__ double s_z[];                 // [kGramTile][kGramStride]
  __shared__ double s_red[kGramThreads];
  const int g = blockIdx.y, tid = threadIdx.x;
  const ure_inter_t* rec = inter[g];
  const long long n = n_rows[g];
  const int E = gram_entries(K);
  const int S = E < kGramThreads ? E : kGramThreads;     // threads per copy
  const int R = kGramThreads / S;                        // copies (1 when E >= 256)
  const int copy = tid / S, slot = tid % S;
  const bool active = copy < R;
  int pa[kGramMaxPer], pb[kGramMaxPer];
  double acc[kGramMaxPer];
#pragma unroll
  for (int j = 0; j < kGramMaxPer; ++j) {
    acc[j] = 0.0;
    pa[j] = pb[j] = 0;
    if (slot + j * S < E) gram_pair(slot + j * S, K, pa[j], pb[j]);
  }
  const int gl = tid % G, rg = tid / G;
  for (long long t0 = (long long)blockIdx.x * kGramTile; t0 < n; t0 += (long long)gridDim.x * kGramTile) {
    for (int rr = rg; rr < kGramTile; rr += RPP) {
      const long long j = t0 + rr;
      const bool valid = j < n;
      int u = 0, it = 0;
      float r = 0.f;
      if (valid) {
        const int4 x = ld_stream_i4(rec + j);
        u = x.x; it = x.y; r = __int_as_float(x.z);
      }
      const float4 pu = valid ? __ldg(reinterpret_cast<const float4*>(P + (size_t)u * D) + gl)
                              : make_float4(0.f, 0.f, 0.f, 0.f);
      double* z = s_z + rr * kGramStride;
      for (int k = 0; k < K; ++k) {
        double dot = 0.0;
        if (valid) {
          const float4 qi = __ldg(reinterpret_cast<const float4*>(Q[k] + (size_t)it * D) + gl);
          dot = (double)pu.x * (double)qi.x;
          dot = fma((double)pu.y, (double)qi.y, dot);
          dot = fma((double)pu.z, (double)qi.z, dot);
          dot = fma((double)pu.w, (double)qi.w, dot);
        }
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o, G);
        if (gl == 0) z[k] = dot;
      }
      if (gl == 0) { z[K] = valid ? 1.0 : 0.0; z[K + 1] = (double)r; }
    }
    __syncthreads();
    if (active) {
      const int tn = n - t0 < kGramTile ? (int)(n - t0) : kGramTile;
      for (int t = copy; t < tn; t += R) {
        const double* z = s_z + t * kGramStride;
#pragma unroll
        for (int j = 0; j < kGramMaxPer; ++j)
          if (slot + j * S < E) acc[j] = fma(z[pa[j]], z[pb[j]], acc[j]);
      }
    }
    __syncthreads();
  }
  double* out = part + ((size_t)g * gridDim.x + blockIdx.x) * E;
  if (R == 1) {
#pragma unroll
    for (int j = 0; j < kGramMaxPer; ++j)
      if (slot + j * S < E) out[slot + j * S] = acc[j];
    return;
  }
  s_red[tid] = active ? acc[0] : 0.0;
  __syncthreads();
  if (tid < E) {
    double s = s_red[tid];
    for (int c = 1; c < R; ++c) s += s_red[c * S + tid];
    out[tid] = s;
  }
}

// out[g][e] = sum over c in CTA order of part[g][c][e]
__global__ void __launch_bounds__(256)
gram_fold_kernel(const double* __restrict__ part, int n_ctas, int E, double* __restrict__ out) {
  const int g = blockIdx.x;
  for (int e = threadIdx.x; e < E; e += blockDim.x) {
    double s = 0.0;
    for (int c = 0; c < n_ctas; ++c) s += part[((size_t)g * n_ctas + c) * E + e];
    out[(size_t)g * E + e] = s;
  }
}

// T[o] = sum_k w[o][k] * Q_k: t = w_0 * q_0, then t = fma(w_k, q_k, t) for k = 1 .. K-1
__global__ void __launch_bounds__(256)
item_wsum_kernel(const float* const* __restrict__ Q, int K, const float* __restrict__ w, int n_out, long long n4,
                 float4* __restrict__ T) {
  const long long total = n4 * n_out;
  for (long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += (long long)gridDim.x * blockDim.x) {
    const int o = (int)(x / n4);
    const long long j = x - (long long)o * n4;
    const float* wo = w + (size_t)o * K;
    float w0 = __ldg(wo);
    float4 q = __ldg(reinterpret_cast<const float4*>(Q[0]) + j);
    float4 s = make_float4(w0 * q.x, w0 * q.y, w0 * q.z, w0 * q.w);
    for (int k = 1; k < K; ++k) {
      const float wk = __ldg(wo + k);
      q = __ldg(reinterpret_cast<const float4*>(Q[k]) + j);
      s.x = fmaf(wk, q.x, s.x); s.y = fmaf(wk, q.y, s.y); s.z = fmaf(wk, q.z, s.z); s.w = fmaf(wk, q.w, s.w);
    }
    T[x] = s;
  }
}

// score[j] = b[s] + P[u].T_s[i] with s = owner[u] (owner -1: the last slot); the dot product in the order of
// ensemble_score_kernel, one group of D/4 lanes per record.  sse += (score - r)^2 in fp64.
template <int D>
__global__ void __launch_bounds__(256)
group_score_kernel(const float* __restrict__ P, const float* __restrict__ T, int n_slots, long long n_item,
                   const float* __restrict__ b, const int32_t* __restrict__ owner, const ure_inter_t* __restrict__ inter,
                   long long n, float* __restrict__ score, double* __restrict__ sse) {
  constexpr int G = D / 4;
  constexpr int GPW = 32 / G;
  const int lane = threadIdx.x & 31;
  const int gl = lane % G;
  const long long n_groups = ((long long)gridDim.x * blockDim.x) / G;
  const long long gid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / G;
  const long long n_round = (n + GPW - 1) / GPW * GPW;
  double acc = 0.0;
  for (long long j = gid; j < n_round; j += n_groups) {
    const bool valid = j < n;
    float dot = 0.f, r = 0.f, bias = 0.f;
    if (valid) {
      const int4 rec = ld_stream_i4(inter + j);
      r = __int_as_float(rec.z);
      const int o = __ldg(owner + rec.x);
      const int s = o >= 0 ? o : n_slots - 1;
      bias = __ldg(b + s);
      const float4 pu = __ldg(reinterpret_cast<const float4*>(P + (size_t)rec.x * D) + gl);
      const float4 qi = __ldg(reinterpret_cast<const float4*>(T + ((size_t)s * n_item + rec.y) * D) + gl);
      dot = pu.x * qi.x;
      dot = fmaf(pu.y, qi.y, dot);
      dot = fmaf(pu.z, qi.z, dot);
      dot = fmaf(pu.w, qi.w, dot);
    }
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o, G);
    if (valid && gl == 0) {
      const float sc = bias + dot;
      if (score) score[j] = sc;
      const float e = sc - r;
      acc += (double)e * (double)e;
    }
  }
  acc = warp_sum(acc);
  __shared__ double part[8];
  if (lane == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0 && sse) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += part[w];
    if (t != 0.0) atomicAdd(sse, t);
  }
}

constexpr size_t kGramSmem = sizeof(double) * kGramTile * kGramStride;    // 68.6 KB: above the 48 KB default

template <int D>
cudaError_t launch_gram(dim3 grid, const float* P, const float* const* Q, int K, const ure_inter_t* const* inter,
                        const int64_t* n, double* part, cudaStream_t st) {
  const cudaError_t e = cudaFuncSetAttribute(combine_gram_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)kGramSmem);
  if (e != cudaSuccess) return e;
  combine_gram_kernel<D><<<grid, kGramThreads, kGramSmem, st>>>(P, Q, K, inter, n, part);
  return cudaGetLastError();
}

bool supported_d(int d) { return d == 8 || d == 16 || d == 32 || d == 64 || d == 128; }

unsigned grid_for(long long work, long long per_block) {
  long long b = (work + per_block - 1) / per_block;
  const long long cap = (long long)num_sms() * 8;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace
}  // namespace ure

extern "C" int ure_combine_gram(const float* d_P, const float* const* d_Q, int n_models, int d,
                                const ure_inter_t* const* d_inter, const int64_t* d_n, int n_groups, double* d_out,
                                double* d_scratch, void* stream) {
  using namespace ure;
  URE_REQUIRE(n_models >= 1 && n_models <= URE_COMBINE_MAX_MODELS, URE_EUNSUPPORTED,
              "ure_combine_gram: n_models=%d not in 1..%d", n_models, URE_COMBINE_MAX_MODELS);
  URE_REQUIRE(supported_d(d), URE_EUNSUPPORTED, "ure_combine_gram: d=%d not in {8,16,32,64,128}", d);
  URE_REQUIRE(n_groups >= 0 && n_groups <= 65535, URE_EINVAL, "ure_combine_gram: n_groups=%d", n_groups);
  if (n_groups == 0) return 0;
  URE_REQUIRE(d_P && d_Q && d_inter && d_n && d_out && d_scratch, URE_EINVAL, "ure_combine_gram: null argument");
  auto st = static_cast<cudaStream_t>(stream);
  const dim3 grid(URE_COMBINE_GRAM_CTAS, (unsigned)n_groups);
  switch (d) {
    case 8: URE_CUDA(launch_gram<8>(grid, d_P, d_Q, n_models, d_inter, d_n, d_scratch, st)); break;
    case 16: URE_CUDA(launch_gram<16>(grid, d_P, d_Q, n_models, d_inter, d_n, d_scratch, st)); break;
    case 32: URE_CUDA(launch_gram<32>(grid, d_P, d_Q, n_models, d_inter, d_n, d_scratch, st)); break;
    case 64: URE_CUDA(launch_gram<64>(grid, d_P, d_Q, n_models, d_inter, d_n, d_scratch, st)); break;
    default: URE_CUDA(launch_gram<128>(grid, d_P, d_Q, n_models, d_inter, d_n, d_scratch, st)); break;
  }
  gram_fold_kernel<<<n_groups, 256, 0, st>>>(d_scratch, URE_COMBINE_GRAM_CTAS, gram_entries(n_models), d_out);
  URE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int ure_item_wsum(const float* const* d_Q, int n_models, const float* d_w, int n_out, int64_t n_item, int d,
                             float* d_T, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_Q && d_w && d_T && n_models >= 1 && n_out >= 0 && n_item >= 0 && d >= 4 && d % 4 == 0, URE_EINVAL,
              "ure_item_wsum: bad argument (n_models=%d n_out=%d n_item=%lld d=%d)", n_models, n_out,
              (long long)n_item, d);
  const long long n4 = n_item * d / 4;
  if (n4 == 0 || n_out == 0) return 0;
  item_wsum_kernel<<<grid_for(n4 * n_out, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      d_Q, n_models, d_w, n_out, n4, reinterpret_cast<float4*>(d_T));
  URE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int ure_group_score(const float* d_P, const float* d_T, int n_slots, int64_t n_item, int d, const float* d_b,
                               const int32_t* d_owner, const ure_inter_t* d_inter, int64_t n, float* d_score,
                               double* d_sse, void* stream) {
  using namespace ure;
  URE_REQUIRE(supported_d(d), URE_EUNSUPPORTED, "ure_group_score: d=%d not in {8,16,32,64,128}", d);
  URE_REQUIRE(n_slots >= 1 && n_item >= 0, URE_EINVAL, "ure_group_score: n_slots=%d n_item=%lld", n_slots,
              (long long)n_item);
  if (n <= 0) return 0;
  URE_REQUIRE(d_P && d_T && d_b && d_owner && d_inter, URE_EINVAL, "ure_group_score: null argument");
  auto st = static_cast<cudaStream_t>(stream);
  const unsigned blocks = grid_for(n, 256 / (d / 4));
  switch (d) {
    case 8: group_score_kernel<8><<<blocks, 256, 0, st>>>(d_P, d_T, n_slots, n_item, d_b, d_owner, d_inter, n, d_score, d_sse); break;
    case 16: group_score_kernel<16><<<blocks, 256, 0, st>>>(d_P, d_T, n_slots, n_item, d_b, d_owner, d_inter, n, d_score, d_sse); break;
    case 32: group_score_kernel<32><<<blocks, 256, 0, st>>>(d_P, d_T, n_slots, n_item, d_b, d_owner, d_inter, n, d_score, d_sse); break;
    case 64: group_score_kernel<64><<<blocks, 256, 0, st>>>(d_P, d_T, n_slots, n_item, d_b, d_owner, d_inter, n, d_score, d_sse); break;
    default: group_score_kernel<128><<<blocks, 256, 0, st>>>(d_P, d_T, n_slots, n_item, d_b, d_owner, d_inter, n, d_score, d_sse); break;
  }
  URE_CUDA(cudaGetLastError());
  return 0;
}
