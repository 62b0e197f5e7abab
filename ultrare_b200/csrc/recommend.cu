// Top-N recommendation over the whole catalogue for a trained or unlearned ensemble.
//
// After the SISA merge every shard model shares one user table, so the ensemble mean (1/K) sum_k P[u].Q_k[i] is
// scale * P[u].S[i] with S = sum_k Q_k and scale = 1/K.  A request of m users is one [m x n_item x d] contraction
// followed by a per-user top-N; the top-N runs in the epilogue, so the score matrix is never written.
//
// topn_kernel (one CTA = 128 requested users x one range of item tiles):
//   all warps   gather the 128 user rows by id and split them into hi / lo tiles (K-major core-matrix layout);
//   warp 0      TMA producer: item tiles of S (the raw fp32 tile is the hi operand: kind::tf32 reads only the top 19
//               bits, DESIGN.md §4.3) and of S_lo = S - trunc_tf32(S), S stages deep;
//   warp 1      MMA issuer: hi*hi + hi*lo + lo*hi into one of two TMEM accumulators (fp32-accurate, as ot_cost.cu);
//   warps 2-5   epilogue, one TMEM lane = one user row per thread: the running top-N of its user in shared memory,
//               a threshold compare per 16 scores, and a cursor through the user's ascending seen list that moves
//               only when a candidate passes the threshold.  The items of a CTA arrive in ascending order, so an equal
//               score never displaces an earlier (smaller) item: ties go to the smaller item id.
// With fewer user tiles than resident CTAs the item range is split over CTAs (a single user still uses every SM);
// each writes a partial list and topn_merge_kernel merges them under the same tie rule.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace ure {
namespace {

constexpr int kRecThreads = 192;       // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue
constexpr int kMaxTopN = 64;
constexpr int kMaxSplits = 256;
constexpr uint32_t kSmemCap = 227u * 1024u;

struct RecLayout {
  uint32_t b_off, b_stage, lo_off, a_hi, a_lo, lbo_a, list_s, list_i, bars, holder, total;
};

__host__ __device__ inline RecLayout rec_layout(int D, int NB, int S, int N) {
  RecLayout L;
  const uint32_t chunks = D / 4;
  uint32_t o = 0;
  L.b_stage = (uint32_t)NB * D * 4 * 2;            // [S tile | S_lo tile]; 1024-byte multiples (swizzle atoms)
  L.lo_off = (uint32_t)NB * D * 4;
  L.b_off = o; o += L.b_stage * S;
  L.lbo_a = kTileRows * 16 + (chunks >= 8 ? 16 : 32);   // padded: the gather's 16-byte stores hit distinct banks
  L.a_hi = o; o += L.lbo_a * chunks;
  L.a_lo = o; o += L.lbo_a * chunks;
  L.list_s = o; o += kTileRows * N * 4;            // [N][128]: entry p of the thread of row r at p * 128 + r
  L.list_i = o; o += kTileRows * N * 4;
  o = (o + 7) / 8 * 8;
  L.bars = o; o += 12 * 8;                         // full[4] empty[4] t_full[2] t_empty[2]
  L.holder = o; o += 16;
  L.total = o;
  return L;
}

// Offer (s, item) to a thread's list (column `ls` / `li` of the [N][128] arrays, sorted by score descending), unless
// the item is in the user's seen list; returns the new threshold (the N-th score).
__device__ __forceinline__ float offer(float s, int item, float* ls, int* li, int N, long long& cur, long long end,
                                    const int32_t* __restrict__ seen) {
  while (cur < end && __ldg(seen + cur) < item) ++cur;
  if (cur < end && __ldg(seen + cur) == item) return ls[(N - 1) * kTileRows];
  int p = N - 1;
  while (p > 0) {
    const float o = ls[(p - 1) * kTileRows];
    if (!(o < s)) break;                           // equal scores keep the earlier, smaller item in front
    ls[p * kTileRows] = o;
    li[p * kTileRows] = li[(p - 1) * kTileRows];
    --p;
  }
  ls[p * kTileRows] = s;
  li[p * kTileRows] = item;
  return ls[(N - 1) * kTileRows];
}

// SW: item tiles arrive as D/32 boxes of {32 floats, NB rows} with the 128-byte swizzle (d >= 32); otherwise as D/4
// boxes of {4 floats, NB rows} that land directly in the no-swizzle core-matrix layout.
template <int D, bool SW>
__global__ void __launch_bounds__(kRecThreads, 1)
topn_kernel(const __grid_constant__ CUtensorMap tm_hi, const __grid_constant__ CUtensorMap tm_lo,
            const float* __restrict__ P, int n_user, const int32_t* __restrict__ users, long long m,
            const long long* __restrict__ seen_off, const int32_t* __restrict__ seen, int n_item, int tiles_per_split,
            int N, float scale, int NB, int S, uint32_t tmem_cols, int32_t* __restrict__ out_items,
            float* __restrict__ out_scores) {
  constexpr int CH = D / 4;
  extern __shared__ __align__(128) unsigned char sm_raw[];
  unsigned char* const sm = sm_raw + ((1024u - (smem_u32(sm_raw) & 1023u)) & 1023u);
  const RecLayout L = rec_layout(D, NB, S, N);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint64_t* const full = reinterpret_cast<uint64_t*>(sm + L.bars);
  uint64_t* const empty = full + 4;
  uint64_t* const t_full = full + 8;
  uint64_t* const t_empty = full + 10;
  uint32_t* const holder = reinterpret_cast<uint32_t*>(sm + L.holder);
  float* const list_s = reinterpret_cast<float*>(sm + L.list_s);
  int* const list_i = reinterpret_cast<int*>(sm + L.list_i);
  const long long row0 = (long long)blockIdx.x * kTileRows;
  const int n_tiles = (n_item + NB - 1) / NB;
  const int t0 = blockIdx.y * tiles_per_split;
  const int t1 = min(n_tiles, t0 + tiles_per_split);
  const int my_tiles = t1 > t0 ? t1 - t0 : 0;

  if (tid == 0) {
    for (int i = 0; i < 4; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], 128); }
    fence_mbar_init();
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_hi) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_lo) : "memory");
  }
  if (warp == 0) tmem_alloc(holder, tmem_cols);
  // ---- the 128 requested user rows -> A_hi / A_lo; rows past m and ids outside the table are zero rows
  for (int idx = tid; idx < kTileRows * CH; idx += kRecThreads) {
    const int r = idx / CH, c = idx % CH;
    const long long row = row0 + r;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < m) {
      const int u = __ldg(users + row);
      if (u >= 0 && u < n_user) v = __ldg(reinterpret_cast<const float4*>(P + (size_t)u * D) + c);
    }
    const float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
    *reinterpret_cast<float4*>(sm + L.a_hi + c * L.lbo_a + r * 16) = hi;
    *reinterpret_cast<float4*>(sm + L.a_lo + c * L.lbo_a + r * 16) =
        make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
  }
  for (int x = tid; x < kTileRows * N; x += kRecThreads) { list_s[x] = -INFINITY; list_i[x] = -1; }
  fence_proxy_async();            // generic-proxy smem writes -> visible to the tensor core (async proxy)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *holder;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0)
      for (int it = 0; it < my_tiles; ++it) {
        const int s = it % S;
        const int i0 = (t0 + it) * NB;
        mbar_wait(&empty[s], (uint32_t)(((it / S) & 1) ^ 1));
        mbar_expect_tx(&full[s], L.b_stage);     // rows past n_item are zero-filled and still counted
        unsigned char* dst = sm + L.b_off + (size_t)s * L.b_stage;
        if (SW) {
#pragma unroll
          for (int a = 0; a < D / 32; ++a) {
            tma_load_2d(dst + a * NB * 128, &tm_hi, 32 * a, i0, &full[s]);
            tma_load_2d(dst + L.lo_off + a * NB * 128, &tm_lo, 32 * a, i0, &full[s]);
          }
        } else {
#pragma unroll
          for (int c = 0; c < CH; ++c) {
            tma_load_2d(dst + c * NB * 16, &tm_hi, 4 * c, i0, &full[s]);
            tma_load_2d(dst + L.lo_off + c * NB * 16, &tm_lo, 4 * c, i0, &full[s]);
          }
        }
      }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      const uint32_t idesc = make_idesc_tf32(NB);
      const uint32_t a_hi = smem_u32(sm + L.a_hi), a_lo = smem_u32(sm + L.a_lo);
      for (int it = 0; it < my_tiles; ++it) {
        const int s = it % S, a = it & 1;
        mbar_wait(&full[s], (uint32_t)((it / S) & 1));
        mbar_wait(&t_empty[a], (uint32_t)(((it >> 1) & 1) ^ 1));
        tc_fence_after();
        const uint32_t b_hi = smem_u32(sm + L.b_off + (size_t)s * L.b_stage), b_lo = b_hi + L.lo_off;
        const uint32_t d = tmem_base + (uint32_t)(a * NB);
#pragma unroll
        for (int kk = 0; kk < D / 8; ++kk) {
          const uint64_t ah = make_desc(a_hi + kk * 2 * L.lbo_a, L.lbo_a, 128);
          const uint64_t al = make_desc(a_lo + kk * 2 * L.lbo_a, L.lbo_a, 128);
          // SW: K atom kk / 4 (NB rows of 128 bytes each), 32 bytes further inside the atom per instruction
          const uint32_t bo = SW ? (uint32_t)((kk >> 2) * NB * 128 + (kk & 3) * 32) : (uint32_t)(kk * 2 * NB * 16);
          const uint64_t bh = SW ? make_desc_sw128(b_hi + bo) : make_desc(b_hi + bo, NB * 16, 128);
          const uint64_t bl = SW ? make_desc_sw128(b_lo + bo) : make_desc(b_lo + bo, NB * 16, 128);
          umma_tf32(d, ah, bh, idesc, kk > 0);
          umma_tf32(d, ah, bl, idesc, 1);
          umma_tf32(d, al, bh, idesc, 1);
        }
        umma_commit(&empty[s]);                  // the item tile may be overwritten by the producer
        umma_commit(&t_full[a]);                 // ... and the accumulator is complete
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue: one user row per thread
    const int rq = warp & 3;
    const int trow = rq * 32 + lane;
    const long long row = row0 + trow;
    const int u = row < m ? __ldg(users + row) : -1;
    const bool valid = u >= 0 && u < n_user;
    long long cur = 0, end = 0;
    if (valid && seen) { cur = __ldg(seen_off + u); end = __ldg(seen_off + u + 1); }
    float* const ls = list_s + trow;
    int* const li = list_i + trow;
    float thr = valid ? -INFINITY : INFINITY;    // rows outside the request take nothing
    for (int it = 0; it < my_tiles; ++it) {
      const int a = it & 1;
      mbar_wait(&t_full[a], (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      const int i0 = (t0 + it) * NB;
      const uint32_t taddr = tmem_base + ((uint32_t)(rq * 32) << 16) + (uint32_t)(a * NB);
      for (int c0 = 0; c0 < NB; c0 += 16) {
        float acc[16];
        __syncwarp();
        tmem_ld16(taddr + (uint32_t)c0, acc);
        float mx = acc[0];
#pragma unroll
        for (int j = 1; j < 16; ++j) mx = fmaxf(mx, acc[j]);
        if (mx * scale > thr) {                  // rare once the list is full: one compare per 16 scores
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float s = acc[j] * scale;
            const int item = i0 + c0 + j;
            if (s > thr && item < n_item) thr = offer(s, item, ls, li, N, cur, end, seen);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&t_empty[a]);
    }
    if (row < m) {
      const long long o = ((long long)blockIdx.y * m + row) * N;
      for (int p = 0; p < N; ++p) {
        out_items[o + p] = li[p * kTileRows];
        out_scores[o + p] = ls[p * kTileRows];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, tmem_cols);
}

__device__ __forceinline__ bool ranks_before(float s, int i, float bs, int bi) { return s > bs || (s == bs && i < bi); }

// partial lists [splits][m][N] -> [m][N]: one warp per user row, N rounds of a warp arg-max over the split heads
__global__ void __launch_bounds__(256)
topn_merge_kernel(const int32_t* __restrict__ p_items, const float* __restrict__ p_scores, long long m, int splits, int N,
                  int32_t* __restrict__ out_items, float* __restrict__ out_scores) {
  __shared__ int head[8][kMaxSplits];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long row = (long long)blockIdx.x * 8 + w;
  if (row >= m) return;
  for (int k = lane; k < splits; k += 32) head[w][k] = 0;
  __syncwarp();
  for (int p = 0; p < N; ++p) {
    float bs = -INFINITY;
    int bi = 0x7fffffff, bk = -1;
    for (int k = lane; k < splits; k += 32) {
      const int h = head[w][k];
      if (h >= N) continue;
      const long long x = ((long long)k * m + row) * N + h;
      const float s = p_scores[x];
      const int i = p_items[x];
      if (bk < 0 || ranks_before(s, i, bs, bi)) { bs = s; bi = i; bk = k; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float os = __shfl_xor_sync(0xffffffffu, bs, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o), ok = __shfl_xor_sync(0xffffffffu, bk, o);
      if (ok >= 0 && (bk < 0 || ranks_before(os, oi, bs, bi))) { bs = os; bi = oi; bk = ok; }
    }
    if (lane == 0) {
      out_items[row * N + p] = bk >= 0 ? bi : -1;
      out_scores[row * N + p] = bk >= 0 ? bs : -INFINITY;
    }
    if (bk >= 0 && (bk & 31) == lane) head[w][bk] += 1;
    __syncwarp();
  }
}

struct TopnPlan {
  int NB, S, splits, tiles_per_split;
  uint32_t tmem_cols;
  size_t smem;
  long long user_tiles;
};

template <int D>
int topn_plan(long long m, long long n_item, int N, TopnPlan* pl) {
  // Widest item tile and deepest pipeline whose footprint leaves room for a second CTA on the SM, else for one
  int NB = 0, S = 0;
  for (uint32_t budget : {kSmemCap / 2 - 1024u, kSmemCap}) {
    for (int nb : {128, 64, 32, 16}) {
      for (int s : {3, 2})
        if (rec_layout(D, nb, s, N).total + 1024 <= budget) { NB = nb; S = s; break; }
      if (NB) break;
    }
    if (NB) break;
  }
  URE_REQUIRE(NB > 0, URE_EUNSUPPORTED, "ure_topn: d=%d top_n=%d does not fit shared memory", D, N);
  pl->NB = NB;
  pl->S = S;
  pl->tmem_cols = 32;
  while ((int)pl->tmem_cols < 2 * NB) pl->tmem_cols <<= 1;
  pl->smem = (size_t)rec_layout(D, NB, S, N).total + 1024;
  const int per_sm_smem = (int)((228u * 1024u) / (pl->smem + 1024));
  int occ = per_sm_smem < 1 ? 1 : per_sm_smem;
  if (occ > 512 / (int)pl->tmem_cols) occ = 512 / (int)pl->tmem_cols;
  pl->user_tiles = (m + kTileRows - 1) / kTileRows;
  const long long item_tiles = (n_item + NB - 1) / NB;
  const long long slots = (long long)num_sms() * occ;
  long long splits = 1;
  if (pl->user_tiles < slots) splits = (slots + pl->user_tiles - 1) / pl->user_tiles;
  if (splits > item_tiles) splits = item_tiles;
  if (splits > kMaxSplits) splits = kMaxSplits;
  const long long per = (item_tiles + splits - 1) / splits;
  pl->tiles_per_split = (int)per;
  pl->splits = (int)((item_tiles + per - 1) / per);
  return 0;
}

int topn_plan_any(int d, long long m, long long n_item, int N, TopnPlan* pl) {
  switch (d) {
    case 8: return topn_plan<8>(m, n_item, N, pl);
    case 16: return topn_plan<16>(m, n_item, N, pl);
    case 32: return topn_plan<32>(m, n_item, N, pl);
    case 64: return topn_plan<64>(m, n_item, N, pl);
    case 128: return topn_plan<128>(m, n_item, N, pl);
    default:
      set_error("ure_topn: d=%d not in {8,16,32,64,128}", d);
      return URE_EUNSUPPORTED;
  }
}

int64_t topn_scratch(const TopnPlan& pl, long long m, int N) {
  return pl.splits > 1 ? (int64_t)pl.splits * m * N * 8 : 0;
}

template <int D>
int launch_topn(const float* P, int n_user, const float* S_hi, const float* S_lo, long long n_item, const int32_t* users,
                long long m, const long long* seen_off, const int32_t* seen, int N, float scale, int32_t* items,
                float* scores, void* scratch, cudaStream_t st) {
  TopnPlan pl;
  if (int rc = topn_plan<D>(m, n_item, N, &pl)) return rc;
  EncodeTiledFn enc = encode_tiled();
  URE_REQUIRE(enc, URE_EUNSUPPORTED, "ure_topn: the driver has no cuTensorMapEncodeTiled");
  constexpr bool kSw = D >= 32;                // a 128-byte swizzle atom is 32 floats of K
  CUtensorMap tm[2];
  const float* src[2] = {S_hi, S_lo};
  for (int x = 0; x < 2; ++x) {
    const cuuint64_t dims[2] = {(cuuint64_t)D, (cuuint64_t)n_item};
    const cuuint64_t strides[1] = {(cuuint64_t)D * 4};
    const cuuint32_t box[2] = {kSw ? 32u : 4u, (cuuint32_t)pl.NB};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(&tm[x], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(src[x]), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, kSw ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    URE_REQUIRE(r == CUDA_SUCCESS, URE_EINVAL, "ure_topn: cuTensorMapEncodeTiled failed (%d)", (int)r);
  }
  auto kern = topn_kernel<D, kSw>;
  URE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
  int32_t* part_items = items;
  float* part_scores = scores;
  if (pl.splits > 1) {
    part_items = static_cast<int32_t*>(scratch);
    part_scores = reinterpret_cast<float*>(part_items + (size_t)pl.splits * m * N);
  }
  kern<<<dim3((unsigned)pl.user_tiles, (unsigned)pl.splits), kRecThreads, pl.smem, st>>>(
      tm[0], tm[1], P, n_user, users, m, seen_off, seen, (int)n_item, pl.tiles_per_split, N, scale, pl.NB, pl.S,
      pl.tmem_cols, part_items, part_scores);
  URE_CUDA(cudaGetLastError());
  if (pl.splits > 1) {
    topn_merge_kernel<<<(unsigned)((m + 7) / 8), 256, 0, st>>>(part_items, part_scores, m, pl.splits, N, items, scores);
    URE_CUDA(cudaGetLastError());
  }
  return 0;
}

// ---------------------------------------------------------------- preparation: S = sum_k Q_k, S_lo = S - trunc(S)
__global__ void item_sum_kernel(const float* const* __restrict__ Q, int K, long long n4, float4* __restrict__ S) {
  for (long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x; x < n4; x += (long long)gridDim.x * blockDim.x) {
    float4 s = __ldg(reinterpret_cast<const float4*>(Q[0]) + x);
    for (int k = 1; k < K; ++k) {
      const float4 q = __ldg(reinterpret_cast<const float4*>(Q[k]) + x);
      s.x += q.x; s.y += q.y; s.z += q.z; s.w += q.w;
    }
    S[x] = s;
  }
}

__global__ void split_lo_kernel(const float4* __restrict__ X, long long n4, float4* __restrict__ lo) {
  for (long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x; x < n4; x += (long long)gridDim.x * blockDim.x) {
    const float4 v = __ldg(X + x);
    lo[x] = make_float4(v.x - tf32_hi(v.x), v.y - tf32_hi(v.y), v.z - tf32_hi(v.z), v.w - tf32_hi(v.w));
  }
}

unsigned stream_blocks(long long n4) {
  long long b = (n4 + 255) / 256;
  const long long cap = (long long)num_sms() * 8;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

// ---------------------------------------------------------------- full-catalogue metrics of the top-N lists
// DCG position weights 1 / log2(p + 2), p < kMaxTopN, as double literals (no fp64 log2 call per thread)
// 1/x for x >= 1 to fp64 accuracy (fp32 seed, three Newton steps) without the fp64 division subroutine, whose call
// made the kernel spill
__device__ __forceinline__ double rcp64(double x) {
  double r = (double)__frcp_rn((float)x);
#pragma unroll
  for (int k = 0; k < 3; ++k) r = fma(r, fma(-x, r, 1.0), r);
  return r;
}
__constant__ double kPosWeight[kMaxTopN] = {
    1.0, 0.6309297535714575, 0.5, 0.43067655807339306,
    0.38685280723454163, 0.3562071871080222, 0.3333333333333333, 0.31546487678572877,
    0.3010299956639812, 0.2890648263178879, 0.27894294565112987, 0.27023815442731974,
    0.26264953503719357, 0.2559580248098155, 0.25, 0.24465054211822604,
    0.23981246656813146, 0.23540891336663824, 0.23137821315975915, 0.227670248696953,
    0.22424382421757544, 0.22106472945750374, 0.21810429198553155, 0.21533827903669653,
    0.21274605355336318, 0.2103099178571525, 0.20801459767650948, 0.20584683246043448,
    0.2037950470905062, 0.20184908658209985, 0.2, 0.19823986317056053,
    0.1965616322328226, 0.1949590218937863, 0.19342640361727081, 0.19195872000656014,
    0.1905514124267734, 0.18920035951687003, 0.18790182470910757, 0.18665241123894338,
    0.1854490234153689, 0.18428883314870617, 0.18316925091363362, 0.18208790046993825,
    0.1810425967800402, 0.18003132665669264, 0.17905223175104137, 0.1781035935540111,
    0.17718382013555792, 0.17629143438888212, 0.17542506358195453, 0.17458343004804494,
    0.17376534287144002, 0.1729696904450771, 0.17219543379409813, 0.17144160057391347,
    0.17070727966372012, 0.16999161628691403, 0.16929380759878143, 0.1686130986895011,
    0.16794877895704194, 0.16730017881017412, 0.16666666666666666, 0.16604764621593782,
};

// One warp per request row: rel = the user's distinct test items with rating >= 4/5 (utils.py:175,180); rows whose
// user has none are not counted.  out += (HR@N, Recall@N, NDCG@N, users).
__global__ void __launch_bounds__(256)
topn_metrics_kernel(const int32_t* __restrict__ items, const int32_t* __restrict__ users, long long m, int N,
                    const ure_inter_t* __restrict__ test, const int32_t* __restrict__ order,
                    const long long* __restrict__ seg, int n_user, double* __restrict__ out) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  double hr = 0.0, recall = 0.0, ndcg = 0.0, cnt = 0.0;
  auto rec = [&](long long x) { return test[order ? order[x] : x]; };
  auto relevant = [](const ure_inter_t& r) { return (double)r.rating >= (4.0 / 5.0); };
  for (long long row = (long long)blockIdx.x * 8 + w; row < m; row += n_warps) {
    const int u = users[row];
    if (u < 0 || u >= n_user) continue;
    const long long b = seg[u], e = seg[u + 1];
    int nrel = 0;
    for (long long x = b + lane; x < e; x += 32) {
      const ure_inter_t r = rec(x);
      if (!relevant(r)) continue;
      bool first = true;                                   // count an item once however often it was rated
      for (long long y = b; y < x && first; ++y) {
        const ure_inter_t q = rec(y);
        first = !(relevant(q) && q.item == r.item);
      }
      nrel += first;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nrel += __shfl_xor_sync(0xffffffffu, nrel, o);
    if (nrel == 0) continue;
    int hits = 0;
    double dcg = 0.0;
    for (int p = lane; p < N; p += 32) {
      const int it = items[row * N + p];
      bool hit = false;
      for (long long y = b; y < e && it >= 0 && !hit; ++y) {
        const ure_inter_t q = rec(y);
        hit = relevant(q) && q.item == it;
      }
      if (hit) { ++hits; dcg += kPosWeight[p]; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) hits += __shfl_xor_sync(0xffffffffu, hits, o);
    dcg = warp_sum(dcg);
    if (lane == 0) {
      double idcg = 0.0;
      for (int p = 0; p < N && p < nrel; ++p) idcg += kPosWeight[p];
      hr += hits > 0 ? 1.0 : 0.0;
      recall += (double)hits * rcp64((double)nrel);
      ndcg += dcg * rcp64(idcg);
      cnt += 1.0;
    }
  }
  __shared__ double part[8][4];
  if (lane == 0) { part[w][0] = hr; part[w][1] = recall; part[w][2] = ndcg; part[w][3] = cnt; }
  __syncthreads();
  if (threadIdx.x < 4) {
    double t = 0.0;
    for (int x = 0; x < 8; ++x) t += part[x][threadIdx.x];
    if (t != 0.0) atomicAdd(out + threadIdx.x, t);
  }
}

}  // namespace
}  // namespace ure

extern "C" int ure_item_sum(const float* const* d_Q, int n_models, int64_t n_item, int d, float* d_S, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_Q && d_S && n_models >= 1 && n_item >= 0 && d >= 4 && d % 4 == 0, URE_EINVAL,
              "ure_item_sum: bad argument (n_models=%d n_item=%lld d=%d)", n_models, (long long)n_item, d);
  const long long n4 = n_item * d / 4;
  if (n4 == 0) return 0;
  item_sum_kernel<<<stream_blocks(n4), 256, 0, static_cast<cudaStream_t>(stream)>>>(d_Q, n_models, n4,
                                                                                  reinterpret_cast<float4*>(d_S));
  URE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int ure_split_lo(const float* d_X, int64_t n, float* d_lo, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_X && d_lo && n >= 0 && n % 4 == 0, URE_EINVAL, "ure_split_lo: bad argument (n=%lld)", (long long)n);
  if (n == 0) return 0;
  split_lo_kernel<<<stream_blocks(n / 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float4*>(d_X), n / 4, reinterpret_cast<float4*>(d_lo));
  URE_CUDA(cudaGetLastError());
  return 0;
}

static int check_topn_shape(int64_t m, int64_t n_item, int d, int top_n) {
  using namespace ure;
  URE_REQUIRE(m >= 0 && n_item >= 1 && n_item < (1ll << 31), URE_EINVAL, "ure_topn: bad shape m=%lld n_item=%lld",
              (long long)m, (long long)n_item);
  URE_REQUIRE(d == 8 || d == 16 || d == 32 || d == 64 || d == 128, URE_EUNSUPPORTED, "ure_topn: d=%d not in {8,16,32,64,128}", d);
  URE_REQUIRE(top_n >= 1 && top_n <= kMaxTopN, URE_EUNSUPPORTED, "ure_topn: top_n=%d not in 1..%d", top_n, kMaxTopN);
  return 0;
}

extern "C" int64_t ure_topn_scratch_bytes(int64_t m, int64_t n_item, int d, int top_n) {
  using namespace ure;
  if (check_topn_shape(m, n_item, d, top_n) || m == 0) return 0;
  TopnPlan pl;
  if (topn_plan_any(d, m, n_item, top_n, &pl)) return 0;
  return topn_scratch(pl, m, top_n);
}

extern "C" int ure_topn(const float* d_P, int n_user, const float* d_S, const float* d_S_lo, int64_t n_item, int d,
                        const int32_t* d_users, int64_t m, const int64_t* d_seen_off, const int32_t* d_seen, int top_n,
                        float scale, int32_t* d_items, float* d_scores, void* d_scratch, void* stream) {
  using namespace ure;
  if (int rc = check_topn_shape(m, n_item, d, top_n)) return rc;
  URE_REQUIRE(d_P && d_S && d_S_lo && n_user >= 1 && (m == 0 || (d_users && d_items && d_scores)), URE_EINVAL,
              "ure_topn: null argument");
  URE_REQUIRE(!d_seen_off == !d_seen, URE_EINVAL, "ure_topn: seen offsets and items go together");
  URE_REQUIRE(scale > 0.f && isfinite(scale), URE_EINVAL, "ure_topn: scale=%g must be positive", (double)scale);
  if (m == 0) return 0;
  TopnPlan pl;
  if (int rc = topn_plan_any(d, m, n_item, top_n, &pl)) return rc;
  URE_REQUIRE(topn_scratch(pl, m, top_n) == 0 || d_scratch, URE_EINVAL, "ure_topn: scratch missing");
  auto st = static_cast<cudaStream_t>(stream);
  auto so = reinterpret_cast<const long long*>(d_seen_off);
  switch (d) {
    case 8: return launch_topn<8>(d_P, n_user, d_S, d_S_lo, n_item, d_users, m, so, d_seen, top_n, scale, d_items, d_scores, d_scratch, st);
    case 16: return launch_topn<16>(d_P, n_user, d_S, d_S_lo, n_item, d_users, m, so, d_seen, top_n, scale, d_items, d_scores, d_scratch, st);
    case 32: return launch_topn<32>(d_P, n_user, d_S, d_S_lo, n_item, d_users, m, so, d_seen, top_n, scale, d_items, d_scores, d_scratch, st);
    case 64: return launch_topn<64>(d_P, n_user, d_S, d_S_lo, n_item, d_users, m, so, d_seen, top_n, scale, d_items, d_scores, d_scratch, st);
    default: return launch_topn<128>(d_P, n_user, d_S, d_S_lo, n_item, d_users, m, so, d_seen, top_n, scale, d_items, d_scores, d_scratch, st);
  }
}

extern "C" int ure_topn_metrics(const int32_t* d_items, const int32_t* d_users, int64_t m, int top_n,
                                const ure_inter_t* d_test, const int32_t* d_order, const int64_t* d_seg, int n_user,
                                double* d_out, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_out && top_n >= 1 && n_user >= 1 && (m == 0 || (d_items && d_users && d_seg)), URE_EINVAL,
              "ure_topn_metrics: bad argument");
  URE_REQUIRE(top_n <= kMaxTopN, URE_EUNSUPPORTED, "ure_topn_metrics: top_n=%d not in 1..%d", top_n, kMaxTopN);
  if (m <= 0) return 0;
  long long blocks = (m + 7) / 8;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  topn_metrics_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      d_items, d_users, m, top_n, d_test, d_order, reinterpret_cast<const long long*>(d_seg), n_user, d_out);
  URE_CUDA(cudaGetLastError());
  return 0;
}
