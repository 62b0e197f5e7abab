// Ensemble scoring and ranking metrics: the arithmetic of baseTest
// (reference method/utils.py:115-187) and computeNDCG/computeDCG (utils.py:190-210).
#include "common.cuh"

namespace ure {
namespace {

// ---------------------------------------------------------------------------
// score[j] = mean_k P_k[u].Q_k[i]   (utils.py:141-145);  sse += (score - r)^2 (utils.py:148)
// A group of D/4 lanes owns one test interaction and walks the K models; when
// consecutive models share the user table (after the SISA merge all do,
// sisa.py:57-58) the user row stays in registers.
// ---------------------------------------------------------------------------
template <int D>
__device__ __forceinline__ void ensemble_score_body(const float* const* __restrict__ Pk, const float* const* __restrict__ Qk,
                                                    int K, const ure_inter_t* __restrict__ inter, long long n, float denom,
                                                    float* __restrict__ score, double* __restrict__ sse) {
  constexpr int G = D / 4;
  const int lane = threadIdx.x & 31;
  const int gl = lane % G;
  const long long n_groups = ((long long)gridDim.x * blockDim.x) / G;
  const long long gid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / G;
  // trip count must be uniform across the warp: round n up to the groups of one warp
  constexpr int GPW = 32 / G;
  const long long n_round = (n + GPW - 1) / GPW * GPW;
  double acc = 0.0;
  for (long long j = gid; j < n_round; j += n_groups) {
    const bool valid = j < n;
    int u = 0, it = 0;
    float r = 0.f;
    if (valid) {
      const int4 rec = ld_stream_i4(inter + j);
      u = rec.x; it = rec.y; r = __int_as_float(rec.z);
    }
    float sum = 0.f;
    const float* lastP = nullptr;
    float4 pu = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = 0; k < K; ++k) {
      const float* P = Pk[k];
      const float* Q = Qk[k];
      float dot = 0.f;
      if (valid) {
        if (P != lastP) { pu = __ldg(reinterpret_cast<const float4*>(P + (size_t)u * D) + gl); lastP = P; }
        const float4 qi = __ldg(reinterpret_cast<const float4*>(Q + (size_t)it * D) + gl);
        dot = pu.x * qi.x;
        dot = fmaf(pu.y, qi.y, dot);
        dot = fmaf(pu.z, qi.z, dot);
        dot = fmaf(pu.w, qi.w, dot);
      }
#pragma unroll
      for (int o = G / 2; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o, G);
      sum += dot;
    }
    if (valid && gl == 0) {
      const float sc = sum / denom;             // torch.stack(preds).mean(0): sum then divide
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

template <int D>
__global__ void __launch_bounds__(256)
ensemble_score_kernel(const float* const* __restrict__ Pk, const float* const* __restrict__ Qk, int K,
                      const ure_inter_t* __restrict__ inter, long long n, float denom,
                      float* __restrict__ score, double* __restrict__ sse) {
  ensemble_score_body<D>(Pk, Qk, K, inter, n, denom, score, sse);
}

// many evaluations in one launch (blockIdx.y = job): the per-epoch in-training evaluations of scratch.py:83-97
template <int D>
__global__ void __launch_bounds__(256)
ensemble_score_jobs_kernel(const ure_eval_job_t* __restrict__ jobs) {
  const ure_eval_job_t jb = jobs[blockIdx.y];
  if (jb.n <= 0) return;
  ensemble_score_body<D>(jb.P, jb.Q, jb.n_models, jb.inter, jb.n, jb.denom, jb.score, jb.out);
}

// ---------------------------------------------------------------------------
// HR@10 / NDCG@10 per user segment, one warp per user (utils.py:166-181).
//   rank_v(e) = #{e' : v(e') > v(e) or (v(e') == v(e) and e' > e)}   ("later index first")
//   where > and == are NumPy's sort order: NaN above +inf and equal to every NaN, -0 == +0 (rank_key)
//   top_pred[p] / top_rating[p] = element of rank p  (p < 10)
//   relevance[p] = r[top_pred[p]] ; hit = relevance >= 4/5 ; HR = #hit / 10
//   common[p] = top_rating[p] in set(top_pred)        (positional, utils.py:179)
//   NDCG = (sum_p relevance[p]*hit[p]*common[p] * w_p) / sum_p w_p,  w_0 = 1, w_p = 1/log2(p+1)
// ---------------------------------------------------------------------------
constexpr int kSegStage = 512;        // a segment up to this long is staged in shared memory (score, rating)
constexpr int kSegCount = 64;         // up to this long: ranks by counting (L * ceil(L / 32) steps); longer: ten arg-max rounds
// DCG position weights 1 / log2(p + 1) (w_0 = 1) and their sum over the top 10, as double literals: fp64 log2 and
// division per thread cost more than the ranking itself on this part
static_assert(URE_TOP_K == 10, "weight table below");
__constant__ double kDcgWeight[URE_TOP_K] = {1.0, 1.0, 0.6309297535714575, 0.5, 0.43067655807339306,
                                             0.38685280723454163, 0.3562071871080222, 0.3333333333333333,
                                             0.31546487678572877, 0.3010299956639812};
constexpr double kIdcg = 5.254494511770457;

// Unsigned key whose order is the order np.sort puts float values in: every NaN maps to the top key (a NaN score ranks
// first, as in argsort(kind='stable')[::-1]), -0 and +0 share a key.  The order on keys is total, so the ranks of a
// segment are a permutation and every slot of the top-10 lists is written exactly once (float comparisons are false for
// NaN: several elements would share a rank and slots would stay unwritten).  Every key is > 0.
// (selects, not branches: branches here keep the compiler from unrolling the staging loop)
__device__ __forceinline__ unsigned rank_key(float v) {
  const unsigned b = __float_as_uint(v);
  const unsigned k = b ^ ((unsigned)((int)b >> 31) | 0x80000000u);      // negative: ~b, positive: b | sign bit
  return v != v ? 0xffffffffu : (v == 0.f ? 0x80000000u : k);
}

// the value of a key (not NaN; -0 comes back as +0): the relevance of a staged rating without another global load
__device__ __forceinline__ float key_value(unsigned k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

__device__ __forceinline__ void rank_metrics_body(const ure_inter_t* __restrict__ inter, const float* __restrict__ score,
                                                  const int32_t* __restrict__ order, const long long* __restrict__ seg,
                                                  long long n_seg, double* __restrict__ out) {
  __shared__ int top_pred[8][URE_TOP_K];
  __shared__ int top_rating[8][URE_TOP_K];
  __shared__ uint2 s_key[8][kSegStage];
  const int lane = threadIdx.x & 31;
  const int w = threadIdx.x >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  // consecutive segments go to DIFFERENT CTAs (warp w of CTA b takes segment w * gridDim.x + b): rating files list their
  // heaviest users next to each other, and eight long segments in one CTA were the tail of the whole kernel
  double ndcg_sum = 0.0, hr_sum = 0.0, users = 0.0;
  const double wgt = lane < URE_TOP_K ? kDcgWeight[lane] : 0.0;
  for (long long sgm = (long long)w * gridDim.x + blockIdx.x; sgm < n_seg; sgm += n_warps) {
    const long long b = seg[sgm];
    const int L = (int)(seg[sgm + 1] - b);
    if (L <= 0) continue;
    if (lane < URE_TOP_K) { top_pred[w][lane] = -1; top_rating[w][lane] = -1; }
    const bool staged = L <= kSegStage;
    auto row_of = [&](int f) { return order ? (long long)order[b + f] : b + f; };
    // rank keys of (score, rating) of element f of the segment: from shared memory, or -- very long segments -- from
    // global memory
    auto staged_key = [&](int f) { return s_key[w][f]; };
    auto global_key = [&](int f) {
      const long long rf = row_of(f);
      return make_uint2(rank_key(score[rf]), rank_key(inter[rf].rating));
    };
    // every lane counts the elements ranked before its own, both orders in one sweep
    auto count_ranks = [&](auto key_of) {
      for (int e = lane; e < L; e += 32) {
        const uint2 me = key_of(e);
        int rp = 0, rr = 0;
        for (int f = 0; f < L; ++f) {
          const uint2 o = key_of(f);
          rp += (o.x > me.x) || (o.x == me.x && f > e);
          rr += (o.y > me.y) || (o.y == me.y && f > e);
        }
        if (rp < URE_TOP_K) top_pred[w][rp] = e;
        if (rr < URE_TOP_K) top_rating[w][rr] = e;
      }
    };
    if (staged)
      for (int e = lane; e < L; e += 32) {
        const long long re = row_of(e);
        s_key[w][e] = make_uint2(rank_key(score[re]), rank_key(inter[re].rating));
      }
    __syncwarp();
    if (staged && L > kSegCount) {
      // the element of rank p is the p-th in the order (value descending, index descending): ten rounds of a warp
      // arg-max over the staged segment instead of L^2 comparisons (one heavy user used to be the kernel's tail)
      // (both orders in one sweep: two independent compare chains per lane instead of twenty dependent rounds)
      unsigned taken_p = 0, taken_r = 0;     // bit k: element lane + 32 k is already placed in that order
      const int P = L < URE_TOP_K ? L : URE_TOP_K;
      for (int p = 0; p < P; ++p) {
        unsigned vp = 0u, vr = 0u;           // below every key: an untaken element always wins its round
        int ep = -1, er = -1;
        for (int k = 0, e = lane; e < L; ++k, e += 32) {
          const uint2 x = s_key[w][e];
          if (!((taken_p >> k) & 1u) && (x.x > vp || (x.x == vp && e > ep))) { vp = x.x; ep = e; }
          if (!((taken_r >> k) & 1u) && (x.y > vr || (x.y == vr && e > er))) { vr = x.y; er = e; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const unsigned ovp = __shfl_xor_sync(0xffffffffu, vp, o), ovr = __shfl_xor_sync(0xffffffffu, vr, o);
          const int oep = __shfl_xor_sync(0xffffffffu, ep, o), oer = __shfl_xor_sync(0xffffffffu, er, o);
          if (ovp > vp || (ovp == vp && oep > ep)) { vp = ovp; ep = oep; }
          if (ovr > vr || (ovr == vr && oer > er)) { vr = ovr; er = oer; }
        }
        if (lane == 0) { top_pred[w][p] = ep; top_rating[w][p] = er; }
        if (ep >= 0 && (ep & 31) == lane) taken_p |= 1u << (ep >> 5);
        if (er >= 0 && (er & 31) == lane) taken_r |= 1u << (er >> 5);
      }
    } else if (staged) {
      // short segments (the common case: a few test rows per user): broadcast reads of shared memory
      count_ranks(staged_key);
    } else {
      // the very long ones that are not staged (a loop of their own: the key arithmetic stays out of the staged one)
      count_ranks(global_key);
    }
    __syncwarp();
    double rel = 0.0, hit = 0.0;
    if (lane < URE_TOP_K && lane < L) {
      const int ep = top_pred[w][lane];
      const double relevance = staged ? key_value(s_key[w][ep].y) : inter[row_of(ep)].rating;
      const bool h = relevance >= (4.0 / 5.0);
      const int tr = top_rating[w][lane];
      bool common = false;
#pragma unroll
      for (int q = 0; q < URE_TOP_K; ++q) common |= (top_pred[w][q] == tr);
      hit = h ? 1.0 : 0.0;
      rel = (h && common) ? relevance * wgt : 0.0;
    }
    rel = warp_sum(rel);
    hit = warp_sum(hit);
    if (lane == 0) {
      ndcg_sum += rel / kIdcg;
      hr_sum += hit / (double)URE_TOP_K;
      users += 1.0;
    }
    __syncwarp();
  }
  // one set of atomics per CTA (thousands of warps on three addresses serialise in L2)
  __shared__ double s_part[8][3];
  if (lane == 0) { s_part[w][0] = ndcg_sum; s_part[w][1] = hr_sum; s_part[w][2] = users; }
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int x = 0; x < 8; ++x) t += s_part[x][threadIdx.x];
    if (t != 0.0) atomicAdd(out + threadIdx.x, t);
  }
}

__global__ void __launch_bounds__(256)
rank_metrics_kernel(const ure_inter_t* __restrict__ inter, const float* __restrict__ score,
                    const int32_t* __restrict__ order, const long long* __restrict__ seg, long long n_seg,
                    double* __restrict__ out) {
  rank_metrics_body(inter, score, order, seg, n_seg, out);
}

__global__ void __launch_bounds__(256)
rank_metrics_jobs_kernel(const ure_eval_job_t* __restrict__ jobs) {
  const ure_eval_job_t jb = jobs[blockIdx.y];
  if (jb.n_seg <= 0 || jb.n <= 0) return;
  rank_metrics_body(jb.inter, jb.score, jb.order, reinterpret_cast<const long long*>(jb.seg), jb.n_seg, jb.out + 1);
}

__global__ void __launch_bounds__(256)
score_finalize_kernel(const float* __restrict__ sum, const ure_inter_t* __restrict__ inter, long long n, float denom,
                      float* __restrict__ score, double* __restrict__ sse) {
  double acc = 0.0;
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x) {
    const float sc = sum[j] / denom;
    score[j] = sc;
    const float e = sc - inter[j].rating;
    acc += (double)e * (double)e;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0 && sse && acc != 0.0) atomicAdd(sse, acc);
}

template <int D>
int launch_score(const float* const* P, const float* const* Q, int K, const ure_inter_t* inter, long long n,
                 float denom, float* score, double* sse, cudaStream_t st) {
  constexpr int G = D / 4;
  const long long groups_per_block = 256 / G;
  long long blocks = (n + groups_per_block - 1) / groups_per_block;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  ensemble_score_kernel<D><<<(unsigned)blocks, 256, 0, st>>>(P, Q, K, inter, n, denom, score, sse);
  URE_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace
}  // namespace ure

extern "C" int ure_ensemble_score(const float* const* d_P, const float* const* d_Q, int n_models, int d,
                                  const ure_inter_t* d_inter, int64_t n, float denom, float* d_score,
                                  double* d_sse, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_P && d_Q && (d_inter || n == 0), URE_EINVAL, "ure_ensemble_score: null argument");
  URE_REQUIRE(n_models >= 1 && denom > 0.f, URE_EINVAL, "ure_ensemble_score: n_models=%d denom=%g", n_models, (double)denom);
  if (n <= 0) return 0;
  auto st = static_cast<cudaStream_t>(stream);
  switch (d) {
    case 8: return launch_score<8>(d_P, d_Q, n_models, d_inter, n, denom, d_score, d_sse, st);
    case 16: return launch_score<16>(d_P, d_Q, n_models, d_inter, n, denom, d_score, d_sse, st);
    case 32: return launch_score<32>(d_P, d_Q, n_models, d_inter, n, denom, d_score, d_sse, st);
    case 64: return launch_score<64>(d_P, d_Q, n_models, d_inter, n, denom, d_score, d_sse, st);
    case 128: return launch_score<128>(d_P, d_Q, n_models, d_inter, n, denom, d_score, d_sse, st);
    default:
      set_error("ure_ensemble_score: d=%d not in {8,16,32,64,128}", d);
      return URE_EUNSUPPORTED;
  }
}

extern "C" int ure_score_finalize(const float* d_sum, const ure_inter_t* d_inter, int64_t n, float denom,
                                  float* d_score, double* d_sse, void* stream) {
  using namespace ure;
  URE_REQUIRE(n == 0 || (d_sum && d_inter && d_score), URE_EINVAL, "ure_score_finalize: null argument");
  URE_REQUIRE(denom > 0.f, URE_EINVAL, "ure_score_finalize: denom=%g", (double)denom);
  if (n <= 0) return 0;
  long long blocks = (n + 255) / 256;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  score_finalize_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_sum, d_inter, n, denom,
                                                                                     d_score, d_sse);
  URE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int ure_rank_metrics(const ure_inter_t* d_inter, const float* d_score, const int32_t* d_order,
                                const int64_t* d_seg, int64_t n_seg, double* d_out, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_out && (n_seg == 0 || (d_inter && d_score && d_seg)), URE_EINVAL,
              "ure_rank_metrics: null argument");
  if (n_seg <= 0) return 0;
  long long blocks = (n_seg + 7) / 8;
  const long long cap = (long long)num_sms() * 4;            // 32 KB of shared memory per CTA: a full wave
  if (blocks > cap) blocks = cap;
  rank_metrics_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      d_inter, d_score, d_order, reinterpret_cast<const long long*>(d_seg), n_seg, d_out);
  URE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int ure_eval_jobs(const ure_eval_job_t* d_jobs, int n_jobs, int d, int64_t max_n, int64_t max_seg,
                             void* stream) {
  using namespace ure;
  URE_REQUIRE(d_jobs && n_jobs >= 0 && n_jobs <= 65535 && max_n >= 0 && max_seg >= 0, URE_EINVAL,
              "ure_eval_jobs: bad argument (n_jobs=%d)", n_jobs);
  if (n_jobs == 0 || max_n == 0) return 0;
  auto st = static_cast<cudaStream_t>(stream);
  // a full wave of CTAs over all jobs together: few blocks per job when there are many jobs
  auto blocks_for = [&](long long want) {
    long long per_job = ((long long)num_sms() * 8 + n_jobs - 1) / n_jobs;
    if (per_job < 1) per_job = 1;
    return (unsigned)(want < per_job ? (want < 1 ? 1 : want) : per_job);
  };
  {
    const int G = d / 4;
    URE_REQUIRE(d == 8 || d == 16 || d == 32 || d == 64 || d == 128, URE_EUNSUPPORTED, "ure_eval_jobs: d=%d not in {8,16,32,64,128}", d);
    const dim3 grid(blocks_for((max_n + 256 / G - 1) / (256 / G)), (unsigned)n_jobs);
    switch (d) {
      case 8: ensemble_score_jobs_kernel<8><<<grid, 256, 0, st>>>(d_jobs); break;
      case 16: ensemble_score_jobs_kernel<16><<<grid, 256, 0, st>>>(d_jobs); break;
      case 32: ensemble_score_jobs_kernel<32><<<grid, 256, 0, st>>>(d_jobs); break;
      case 64: ensemble_score_jobs_kernel<64><<<grid, 256, 0, st>>>(d_jobs); break;
      default: ensemble_score_jobs_kernel<128><<<grid, 256, 0, st>>>(d_jobs); break;
    }
  }
  if (max_seg > 0) {
    const dim3 grid(blocks_for((max_seg + 7) / 8), (unsigned)n_jobs);
    rank_metrics_jobs_kernel<<<grid, 256, 0, st>>>(d_jobs);
  }
  URE_CUDA(cudaGetLastError());
  return 0;
}
