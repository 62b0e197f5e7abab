// Balanced-OT user grouping: Sinkhorn scaling, plan, assignment and centroid sums.
//
// Replaces the ot.emd call and the label/centroid lines of ot_cluster (reference
// method/utils.py:641-648).  The reference's comment says "compute sinkhorn distance"
// but the code calls the exact network simplex (SURVEY.md §0.2); north_star mandates
// Sinkhorn on the GPU, whose eps -> 0 limit is that exact plan.
//
// With uniform row marginals a_i = 1/n the row potential is a function of the column
// potentials g alone, so one Sinkhorn iteration is ONE streaming pass over the cost
// matrix M [n, kpad] (row major, columns >= k hold +inf):
//     t_ij = (g_j - M_ij)/eps ;  P_ij = a_i * softmax_j(t_ij) ;  colsum_j = sum_i P_ij
//     g_j += eps * (log b_j - log colsum_j),  b_j = 1/k
// Row work is a warp-shuffle reduction over kpad/4 lanes.  The column sums are accumulated in the LOG DOMAIN
// (extended exponent): every lane keeps, per column, a reference exponent r (an integer, re-based when an
// entry lies more than 2^60 above it) and the sum of 2^(t_ij - rowLSE_i - r) -- so a column whose every entry is
// hundreds of binades below its row maximum (stale warm-start potentials at a small eps) still has an exact,
// non-zero sum, exactly as the float64 log-sum-exp of oracle/ot.py:sinkhorn_log.  One MUFU ex2 per element:
// the same exponential feeds the row sum (times 2^r, a per-lane constant) and the column sum.  Partial sums
// travel as (r, s) pairs: lanes -> warp (shuffle) -> CTA (shared memory, fixed order) -> grid (one fp64 atomic
// per column and CTA of s * 2^r / n, r clamped at -960; the cluster form keeps the pairs to the end).
#include "common.cuh"
#include <cooperative_groups.h>

namespace ure {
namespace {

constexpr float kNoRef = -1.0e30f;        // reference exponent of a column that has not seen a finite entry yet
constexpr float kRebase = 60.f;           // an entry more than this many binades above the reference re-bases it
constexpr float kMinExp = -960.f;         // smallest exponent a partial sum is converted to fp64 with

constexpr float kLog2e = 1.4426950408889634f;

// 2^x for x <= 0 (after the max shift): one MUFU, flush-to-zero; relative error 2^-22
__device__ __forceinline__ float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
constexpr int kMaxStages = 16;
constexpr int kSkThreads = 512;

template <int KPAD>
struct RowMap {
  static constexpr int LPR = (KPAD / 4 < 32) ? KPAD / 4 : 32;   // lanes per row
  static constexpr int VEC = KPAD / 4 / LPR;                     // float4 per lane
  static constexpr int RPW = 32 / LPR;                           // rows per warp pass
};

// softmax numerators of one row fragment; returns 1/sum over the row (group reduction)
template <int KPAD>
__device__ __forceinline__ float row_softmax(const float4 (&m)[RowMap<KPAD>::VEC], const float4 (&g)[RowMap<KPAD>::VEC],
                                             float scale, float4 (&p)[RowMap<KPAD>::VEC], float& row_max_t) {
  using RM = RowMap<KPAD>;
  float mx = -INFINITY;
#pragma unroll
  for (int v = 0; v < RM::VEC; ++v) {
    p[v].x = (g[v].x - m[v].x) * scale; p[v].y = (g[v].y - m[v].y) * scale;
    p[v].z = (g[v].z - m[v].z) * scale; p[v].w = (g[v].w - m[v].w) * scale;
    mx = fmaxf(mx, fmaxf(fmaxf(p[v].x, p[v].y), fmaxf(p[v].z, p[v].w)));
  }
#pragma unroll
  for (int o = RM::LPR / 2; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o, RM::LPR));
  float s = 0.f;
#pragma unroll
  for (int v = 0; v < RM::VEC; ++v) {
    p[v].x = ex2_fast(p[v].x - mx); p[v].y = ex2_fast(p[v].y - mx);
    p[v].z = ex2_fast(p[v].z - mx); p[v].w = ex2_fast(p[v].w - mx);
    s += (p[v].x + p[v].y) + (p[v].z + p[v].w);
  }
#pragma unroll
  for (int o = RM::LPR / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, RM::LPR);
  row_max_t = mx;
  return __frcp_rn(s);                     // s in [1, KPAD]
}

template <int KPAD>
__device__ __forceinline__ void load_g(const float* g, int k, int gl, float4 (&out)[RowMap<KPAD>::VEC]) {
  using RM = RowMap<KPAD>;
#pragma unroll
  for (int v = 0; v < RM::VEC; ++v) {
    const int c = (v * RM::LPR + gl) * 4;
    out[v].x = c + 0 < k ? g[c + 0] : 0.f; out[v].y = c + 1 < k ? g[c + 1] : 0.f;
    out[v].z = c + 2 < k ? g[c + 2] : 0.f; out[v].w = c + 3 < k ? g[c + 3] : 0.f;
  }
}

// Column sums of rows [r0,r1) handled by this CTA, in the log domain: every warp leaves, per column, the pair
// (r, s) with sum_i P_ij * n = s * 2^r in part_r / part_s [n_warps][KPAD] (plain stores; the caller folds the
// warps with fold_parts after a __syncthreads).  Msrc: row-major matrix base (global or shared) whose row 0 is
// row `base_row`.  Arithmetic in log2 units: t = (g_j - M_ij) * log2(e)/eps.
template <int KPAD>
__device__ __forceinline__ void colsum_rows(const float* Msrc, long long base_row, long long r0, long long r1,
                                            const float* g_sh, int k, float scale, float* part_r, float* part_s,
                                            int stride = KPAD) {       // floats between rows (>= KPAD: a column slice)
  using RM = RowMap<KPAD>;
  const int lane = threadIdx.x & 31;
  const int gl = lane % RM::LPR;
  const int rw = lane / RM::LPR;
  const int warp = threadIdx.x >> 5;
  const int n_warps = blockDim.x >> 5;
  float4 gs[RM::VEC], ref[RM::VEC], cref[RM::VEC], acc[RM::VEC];
  load_g<KPAD>(g_sh, k, gl, gs);
#pragma unroll
  for (int v = 0; v < RM::VEC; ++v) {
    gs[v].x *= scale; gs[v].y *= scale; gs[v].z *= scale; gs[v].w *= scale;
    ref[v] = make_float4(kNoRef, kNoRef, kNoRef, kNoRef);
    cref[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float nscale = -scale;
#pragma unroll 2
  for (long long row0 = r0 + (long long)warp * RM::RPW; row0 < r1; row0 += (long long)n_warps * RM::RPW) {
    const long long row = row0 + rw;
    const bool valid = row < r1;
    float4 t[RM::VEC];
    float mx = -1.0e30f;                     // a row slot past the end holds +inf costs: every q below is exactly 0
#pragma unroll
    for (int v = 0; v < RM::VEC; ++v) {
      float4 m = make_float4(INFINITY, INFINITY, INFINITY, INFINITY);
      if (valid) m = *(reinterpret_cast<const float4*>(Msrc + (row - base_row) * stride) + v * RM::LPR + gl);
      t[v].x = fmaf(m.x, nscale, gs[v].x); t[v].y = fmaf(m.y, nscale, gs[v].y);
      t[v].z = fmaf(m.z, nscale, gs[v].z); t[v].w = fmaf(m.w, nscale, gs[v].w);
      mx = fmaxf(mx, fmaxf(fmaxf(t[v].x, t[v].y), fmaxf(t[v].z, t[v].w)));
    }
#pragma unroll
    for (int o = RM::LPR / 2; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o, RM::LPR));
    // q = 2^((t - rowmax) - r): the entry relative to the lane's column reference.  One exponential per element; a
    // q beyond 2^60 (the first row of a column, or a jump of more than 60 binades) re-bases the reference first.
    float4 q[RM::VEC];
    float big = 0.f;
#pragma unroll
    for (int v = 0; v < RM::VEC; ++v) {
      q[v].x = ex2_fast((t[v].x - mx) - ref[v].x); q[v].y = ex2_fast((t[v].y - mx) - ref[v].y);
      q[v].z = ex2_fast((t[v].z - mx) - ref[v].z); q[v].w = ex2_fast((t[v].w - mx) - ref[v].w);
      big = fmaxf(big, fmaxf(fmaxf(q[v].x, q[v].y), fmaxf(q[v].z, q[v].w)));
    }
    if (big > 1.0e18f) {                     // rare
#pragma unroll
      for (int v = 0; v < RM::VEC; ++v) {
#define URE_REBASE(C)                                                     \
  if (q[v].C > 1.0e18f) {                                                 \
    const float nr = rintf(t[v].C - mx);                                  \
    acc[v].C *= ex2_fast(ref[v].C - nr);                                  \
    ref[v].C = nr;                                                        \
    cref[v].C = ex2_fast(nr);                                             \
    q[v].C = ex2_fast((t[v].C - mx) - nr);                                \
  }
        URE_REBASE(x) URE_REBASE(y) URE_REBASE(z) URE_REBASE(w)
#undef URE_REBASE
      }
    }
    float s = 0.f;
#pragma unroll
    for (int v = 0; v < RM::VEC; ++v) {      // the row sum wants 2^(t - rowmax) = q * 2^r
      s = fmaf(q[v].x, cref[v].x, s); s = fmaf(q[v].y, cref[v].y, s);
      s = fmaf(q[v].z, cref[v].z, s); s = fmaf(q[v].w, cref[v].w, s);
    }
#pragma unroll
    for (int o = RM::LPR / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, RM::LPR);
    const float w = valid ? __frcp_rn(s) : 0.f;      // s in [1, KPAD] for a valid row (its maximum contributes 1)
#pragma unroll
    for (int v = 0; v < RM::VEC; ++v) {
      acc[v].x = fmaf(q[v].x, w, acc[v].x); acc[v].y = fmaf(q[v].y, w, acc[v].y);
      acc[v].z = fmaf(q[v].z, w, acc[v].z); acc[v].w = fmaf(q[v].w, w, acc[v].w);
    }
  }
  // lanes with equal gl hold the same columns: fold the RPW row slots of the warp, re-based to the larger reference
#pragma unroll
  for (int v = 0; v < RM::VEC; ++v) {
#pragma unroll
    for (int o = RM::LPR; o < 32; o <<= 1) {
#define URE_FOLD(C)                                                                     \
  {                                                                                     \
    const float r2 = __shfl_xor_sync(0xffffffffu, ref[v].C, o);                         \
    const float a2 = __shfl_xor_sync(0xffffffffu, acc[v].C, o);                         \
    const float R = fmaxf(ref[v].C, r2);                                                \
    acc[v].C = acc[v].C * ex2_fast(ref[v].C - R) + a2 * ex2_fast(r2 - R);               \
    ref[v].C = R;                                                                       \
  }
      URE_FOLD(x) URE_FOLD(y) URE_FOLD(z) URE_FOLD(w)
#undef URE_FOLD
    }
    if (rw == 0) {
      const int c = (v * RM::LPR + gl) * 4;
      *reinterpret_cast<float4*>(part_r + warp * KPAD + c) = ref[v];
      *reinterpret_cast<float4*>(part_s + warp * KPAD + c) = acc[v];
    }
  }
}

// (r, s) of column j over the CTA's warps, in warp order (deterministic)
__device__ __forceinline__ void fold_parts(const float* part_r, const float* part_s, int n_warps, int kpad, int j,
                                           float& R, float& S) {
  R = kNoRef;
  for (int w = 0; w < n_warps; ++w) R = fmaxf(R, part_r[w * kpad + j]);
  S = 0.f;
  for (int w = 0; w < n_warps; ++w) S = fmaf(part_s[w * kpad + j], ex2_fast(part_r[w * kpad + j] - R), S);
}

// s * 2^r / n as a double (r is an integer; below kMinExp the value is clamped, still positive)
__device__ __forceinline__ double pair_to_double(float R, float S, double a) {
  return ldexp((double)S, (int)fmaxf(R, kMinExp)) * a;
}

// --------------------------------------------------------------------------- split-phase kernels
template <int KPAD>
__global__ void __launch_bounds__(kSkThreads)
colsum_kernel(const float* __restrict__ M, long long n, int k, const float* __restrict__ g, float scale, double a,
              double* __restrict__ colsum, int stride) {
  __shared__ float g_sh[KPAD];
  __shared__ __align__(16) float part_r[(kSkThreads / 32) * KPAD];
  __shared__ __align__(16) float part_s[(kSkThreads / 32) * KPAD];
  for (int j = threadIdx.x; j < KPAD; j += blockDim.x) g_sh[j] = j < k ? g[j] : 0.f;
  __syncthreads();
  const long long per = (n + gridDim.x - 1) / gridDim.x;
  const long long r0 = per * blockIdx.x;
  const long long r1 = r0 + per < n ? r0 + per : n;
  if (r0 >= r1) return;
  colsum_rows<KPAD>(M, 0, r0, r1, g_sh, k, scale, part_r, part_s, stride);
  __syncthreads();
  for (int j = threadIdx.x; j < k; j += blockDim.x) {
    float R, S;
    fold_parts(part_r, part_s, kSkThreads / 32, KPAD, j, R, S);
    if (S != 0.f) atomicAdd(colsum + j, pair_to_double(R, S, a));      // NaN != 0: a poisoned column propagates
  }
}

__global__ void update_g_kernel(float* g, double* colsum, int k, float eps) {
  const int j = threadIdx.x;
  if (j < k) {
    const double c = colsum[j];
    g[j] = (float)((double)g[j] + (double)eps * (-log((double)k) - log(c)));
    colsum[j] = 0.0;
  }
}

// --------------------------------------------------------------------------- persistent Sinkhorn, rows of M in shared memory
struct SkStages {
  float eps[kMaxStages];
  int iters[kMaxStages];
  int n;
  float tol;   // a stage ends early once max_j |colsum_j - 1/k| * k < tol (0: always run all iterations)
};
struct SkWorkspace {
  unsigned barrier;
  unsigned pad[31];
  double colsum[3][256];
  double col_err;       // max_j |colsum_j - 1/k| * k seen at the last iteration
  long long iters_done;
};

template <int KPAD>
__global__ void __launch_bounds__(kSkThreads, 1)
sinkhorn_kernel(const float* __restrict__ M, long long n, int k, float* __restrict__ g_io, SkStages stages,
                SkWorkspace* ws) {
  extern __shared__ __align__(16) float m_sh[];     // part_r | part_s [warps][KPAD], then this CTA's rows of M
  __shared__ float g_sh[KPAD];
  constexpr int NWARP = kSkThreads / 32;
  float* const part_r = m_sh;
  float* const part_s = m_sh + NWARP * KPAD;
  float* const rows_sh = m_sh + 2 * NWARP * KPAD;
  const int tid = threadIdx.x;
  const long long per = (n + gridDim.x - 1) / gridDim.x;
  const long long r0 = per * blockIdx.x < n ? per * blockIdx.x : n;
  const long long r1 = r0 + per < n ? r0 + per : n;
  for (int j = tid; j < KPAD; j += blockDim.x) g_sh[j] = j < k ? g_io[j] : 0.f;
  const long long cnt4 = (r1 - r0) * (KPAD / 4);
  const float4* src = reinterpret_cast<const float4*>(M + r0 * KPAD);
  for (long long x = tid; x < cnt4; x += blockDim.x) reinterpret_cast<float4*>(rows_sh)[x] = __ldg(src + x);
  __syncthreads();
  const double a = 1.0 / (double)n;
  const double logb = -log((double)k);
  unsigned bar_target = 0;
  long long it_global = 0;
  for (int s = 0; s < stages.n; ++s) {
    const float eps = stages.eps[s];
    const float scale = kLog2e / eps;
    for (int it = 0; it < stages.iters[s]; ++it, ++it_global) {
      double* cs = ws->colsum[it_global % 3];
      if (r0 < r1) {
        colsum_rows<KPAD>(rows_sh, r0, r0, r1, g_sh, k, scale, part_r, part_s);
        __syncthreads();
        for (int j = tid; j < k; j += blockDim.x) {
          float R, S;
          fold_parts(part_r, part_s, NWARP, KPAD, j, R, S);
          if (S != 0.f) atomicAdd(cs + j, pair_to_double(R, S, a));
        }
      }
      grid_barrier(&ws->barrier, bar_target);
      // every CTA applies the identical update to its private copy of g (and takes the identical
      // early-exit decision: all read the same column sums)
      __shared__ float err_sh;
      if (tid == 0) err_sh = 0.f;
      __syncthreads();
      for (int j = tid; j < k; j += blockDim.x) {
        const double c = __ldcg(cs + j);
        g_sh[j] = (float)((double)g_sh[j] + (double)eps * (logb - log(c)));
        if (blockIdx.x == 0) ws->colsum[(it_global + 2) % 3][j] = 0.0;
        const float e = (float)(fabs(c * (double)k - 1.0));
        atomicMax(reinterpret_cast<int*>(&err_sh), __float_as_int(e));       // e >= 0: int order == float order
      }
      __syncthreads();
      const float err = err_sh;
      if (blockIdx.x == 0 && tid == 0) { ws->col_err = (double)err; ws->iters_done = it_global + 1; }
      __syncthreads();
      if (stages.tol > 0.f && err < stages.tol) { ++it_global; break; }
    }
  }
  if (blockIdx.x == 0)
    for (int j = tid; j < k; j += blockDim.x) g_io[j] = g_sh[j];
}

// --------------------------------------------------------------------------- multi-GPU Sinkhorn over peer memory
// Users (rows of M) are sharded over the GPUs of one NVSwitch domain; an iteration needs the k column sums of ALL
// rows.  Instead of `column pass -> NCCL all-reduce -> update` (three launches and a collective per iteration, each
// costing more than the pass itself at 1 M users per GPU), ONE persistent kernel per GPU runs every iteration:
//   column pass over the GPU's rows -> grid barrier -> CTA 0 stores the GPU's k sums into EVERY peer's exchange
//   buffer (NVLink stores into symmetric memory), fences, and raises its flag there -> every CTA polls the flags in
//   its OWN buffer, adds the per-GPU sums in rank order (identical on every GPU, bit for bit) and updates g.
// Buffers alternate by iteration parity: a peer can only be two iterations ahead after it has seen this GPU's flag of
// the next iteration, which is raised after every CTA here has read the current slot.  Flags only grow (call_base +
// iteration), so nothing is ever reset between calls.  A poll that does not succeed within ~2 s raises the error word
// instead of hanging the GPU.
constexpr int kPeerMax = 16;
struct SkPeers {
  unsigned long long* xchg[kPeerMax];      // every rank's exchange buffer (peer-mapped), this rank's own included
};
struct SkXchg {
  unsigned long long flag[2][kPeerMax];
  double val[2][kPeerMax][256];
};

__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// two CTAs per SM (<= 64 registers): one CTA of 16 warps per SM streams at a third of the HBM rate
template <int KPAD>
__global__ void __launch_bounds__(kSkThreads, 2)
sinkhorn_peer_kernel(const float* __restrict__ M, long long n, double n_total, int k, float* __restrict__ g_io,
                     SkStages stages, SkWorkspace* ws, SkPeers peers, int rank, int world, unsigned long long call_base,
                     int stride) {
  constexpr int NWARP = kSkThreads / 32;
  __shared__ float g_sh[KPAD];
  __shared__ __align__(16) float part_r[NWARP * KPAD];
  __shared__ __align__(16) float part_s[NWARP * KPAD];
  __shared__ float err_sh;
  __shared__ int fail_sh;
  const int tid = threadIdx.x;
  const long long per = (n + gridDim.x - 1) / gridDim.x;
  const long long r0 = per * blockIdx.x < n ? per * blockIdx.x : n;
  const long long r1 = r0 + per < n ? r0 + per : n;
  for (int j = tid; j < KPAD; j += blockDim.x) g_sh[j] = j < k ? g_io[j] : 0.f;
  if (tid == 0) fail_sh = 0;
  __syncthreads();
  const double a = 1.0 / n_total;
  const double logb = -log((double)k);
  SkXchg* const mine = reinterpret_cast<SkXchg*>(peers.xchg[rank]);
  unsigned bar_target = 0;
  long long it_global = 0;
  for (int s = 0; s < stages.n; ++s) {
    const float eps = stages.eps[s];
    const float scale = kLog2e / eps;
    for (int it = 0; it < stages.iters[s]; ++it, ++it_global) {
      double* cs = ws->colsum[it_global % 3];
      const int par = (int)(it_global & 1);
      const unsigned long long stamp = call_base + (unsigned long long)it_global + 1ull;
      if (r0 < r1) {
        colsum_rows<KPAD>(M, 0, r0, r1, g_sh, k, scale, part_r, part_s, stride);
        __syncthreads();
        for (int j = tid; j < k; j += blockDim.x) {
          float R, S;
          fold_parts(part_r, part_s, NWARP, KPAD, j, R, S);
          if (S != 0.f) atomicAdd(cs + j, pair_to_double(R, S, a));
        }
      }
      grid_barrier(&ws->barrier, bar_target);
      if (blockIdx.x == 0) {
        // this GPU's sums -> slot `rank` of every GPU's buffer, then the flag (release, system scope)
        for (int x = tid; x < world * k; x += blockDim.x) {
          const int p = x / k, j = x - p * k;
          reinterpret_cast<SkXchg*>(peers.xchg[p])->val[par][rank][j] = __ldcg(cs + j);
        }
        __threadfence_system();
        __syncthreads();
        if (tid < world) st_release_sys_u64(&reinterpret_cast<SkXchg*>(peers.xchg[tid])->flag[par][rank], stamp);
        for (int j = tid; j < k; j += blockDim.x) ws->colsum[(it_global + 2) % 3][j] = 0.0;
      }
      if (tid < world) {                    // every CTA polls its OWN GPU's flags: one lane per source rank
        long long spins = 0;
        while (ld_acquire_sys_u64(&mine->flag[par][tid]) < stamp)
          if (++spins > (1ll << 23)) { fail_sh = 1; break; }     // a few seconds
      }
      if (tid == 0) err_sh = 0.f;
      __syncthreads();
      if (fail_sh) {                        // a peer never arrived: stop (identical data is not guaranteed any more)
        if (tid == 0) ws->iters_done = -1;
        return;
      }
      for (int j = tid; j < k; j += blockDim.x) {
        double c = 0.0;
        for (int r = 0; r < world; ++r) c += __ldcv(&mine->val[par][r][j]);      // rank order: same sum everywhere
        g_sh[j] = (float)((double)g_sh[j] + (double)eps * (logb - log(c)));
        const float e = (float)(fabs(c * (double)k - 1.0));
        atomicMax(reinterpret_cast<int*>(&err_sh), __float_as_int(e));
      }
      __syncthreads();
      const float err = err_sh;
      if (blockIdx.x == 0 && tid == 0) { ws->col_err = (double)err; ws->iters_done = it_global + 1; }
      __syncthreads();
      if (stages.tol > 0.f && err < stages.tol) { ++it_global; break; }
    }
  }
  if (blockIdx.x == 0)
    for (int j = tid; j < k; j += blockDim.x) g_io[j] = g_sh[j];
}

// --------------------------------------------------------------------------- cluster Sinkhorn (small problems)
// ml1m-sized grouping (n = 6040, k = 5: M is 386 KB) is pure latency: a grid barrier on 148 SMs per iteration
// costs more than the iteration.  Here ONE thread-block cluster holds M in the shared memory of its CTAs, every CTA
// pushes its k partial column sums -- (r, s) pairs -- into every peer's shared memory (distributed shared memory)
// and a hardware cluster barrier ends the iteration; slot arrays alternate, so one barrier per iteration is enough.
constexpr int kClusterMax = 8;

template <int KPAD, int KS>                 // KS <= KPAD columns are kept in shared memory (k <= KS)
__global__ void __launch_bounds__(kSkThreads, 1)
sinkhorn_cluster_kernel(const float* __restrict__ M, long long n, int k, float* __restrict__ g_io, SkStages stages,
                        SkWorkspace* ws) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank(), CS = (int)cluster.num_blocks();
  extern __shared__ __align__(16) float m_sh[];     // this CTA's rows of M
  constexpr int NWARP = kSkThreads / 32;
  __shared__ float g_sh[KS];
  __shared__ __align__(16) float part_r[NWARP * KS];
  __shared__ __align__(16) float part_s[NWARP * KS];
  __shared__ float2 slots[2][kClusterMax][KS];     // [parity][source CTA][column] = (r, s)
  __shared__ float err_sh;
  const int tid = threadIdx.x;
  const long long per = (n + CS - 1) / CS;
  const long long r0 = per * rank < n ? per * rank : n;
  const long long r1 = r0 + per < n ? r0 + per : n;
  for (int j = tid; j < KS; j += blockDim.x) g_sh[j] = j < k ? g_io[j] : 0.f;
  for (int x = tid; x < NWARP * KS; x += blockDim.x) { part_r[x] = kNoRef; part_s[x] = 0.f; }
  {
    const int cnt4 = (int)(r1 - r0) * (KS / 4);
    const float4* src = reinterpret_cast<const float4*>(M + r0 * KPAD);
    for (int x = tid; x < cnt4; x += blockDim.x)
      reinterpret_cast<float4*>(m_sh)[x] = __ldg(src + (x / (KS / 4)) * (KPAD / 4) + x % (KS / 4));
  }
  cluster.sync();                                    // every CTA of the cluster is running: its shared memory exists
  const double log_a = -log((double)n);
  const double logb = -log((double)k);
  long long it_global = 0;
  float last_err = 0.f;
  for (int s = 0; s < stages.n; ++s) {
    const float eps = stages.eps[s];
    const float scale = kLog2e / eps;
    for (int it = 0; it < stages.iters[s]; ++it, ++it_global) {
      const int par = (int)(it_global & 1);
      if (r0 < r1) colsum_rows<KS>(m_sh, r0, r0, r1, g_sh, k, scale, part_r, part_s);   // every warp writes its slot
      __syncthreads();
      if (tid < KS) {
        float R, S;
        fold_parts(part_r, part_s, NWARP, KS, tid, R, S);
        for (int r = 0; r < CS; ++r) *cluster.map_shared_rank(&slots[par][rank][tid], r) = make_float2(R, S);
      }
      if (tid == 0) err_sh = 0.f;
      cluster.sync();                                // all partial sums of this iteration have landed everywhere
      if (tid < k) {
        float Rm = kNoRef;
        for (int r = 0; r < CS; ++r) Rm = fmaxf(Rm, slots[par][r][tid].x);
        double c = 0.0;
        for (int r = 0; r < CS; ++r)                                           // same order in every CTA
          c += (double)slots[par][r][tid].y * (double)ex2_fast(slots[par][r][tid].x - Rm);
        // log of the column sum with the exponent kept apart: no floor, no underflow
        const double logc = log(c) + (double)Rm * 0.6931471805599453 + log_a;
        g_sh[tid] = (float)((double)g_sh[tid] + (double)eps * (logb - logc));
        const float e = (float)(fabs(exp(logc - logb) - 1.0));
        atomicMax(reinterpret_cast<int*>(&err_sh), __float_as_int(e));       // e >= 0: int order == float order
      }
      __syncthreads();
      const float err = err_sh;
      last_err = err;
      if (stages.tol > 0.f && err < stages.tol) { ++it_global; break; }      // identical decision in every CTA
    }
  }
  if (rank == 0) {
    for (int j = tid; j < k; j += blockDim.x) g_io[j] = g_sh[j];
    if (tid == 0) { ws->col_err = (double)last_err; ws->iters_done = it_global; }
  }
  cluster.sync();                                    // no CTA leaves while a peer may still write into it
}

template <int KPAD, int KS>
int launch_sinkhorn_cluster(const float* M, long long n, int k, float* g, const SkStages& st, SkWorkspace* ws, int cs,
                            size_t smem, cudaStream_t stream) {
  auto kern = sinkhorn_cluster_kernel<KPAD, KS>;
  URE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(cs);
  cfg.blockDim = dim3(kSkThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  URE_CUDA(cudaLaunchKernelEx(&cfg, kern, M, n, k, g, st, ws));
  return 0;
}

// --------------------------------------------------------------------------- plan / assignment
template <int KPAD>
__global__ void __launch_bounds__(256)
plan_kernel(const float* __restrict__ M, long long n, int k, const float* __restrict__ g, float scale, float a,
            float* __restrict__ plan) {
  using RM = RowMap<KPAD>;
  __shared__ float g_sh[KPAD];
  for (int j = threadIdx.x; j < KPAD; j += blockDim.x) g_sh[j] = j < k ? g[j] : 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, gl = lane % RM::LPR, rw = lane / RM::LPR;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  float4 gv[RM::VEC];
  load_g<KPAD>(g_sh, k, gl, gv);
  for (long long row0 = warp * RM::RPW; row0 < n; row0 += n_warps * RM::RPW) {
    const long long row = row0 + rw;
    const bool valid = row < n;
    float4 m[RM::VEC], p[RM::VEC];
#pragma unroll
    for (int v = 0; v < RM::VEC; ++v) {
      m[v] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (valid) m[v] = __ldg(reinterpret_cast<const float4*>(M + row * KPAD) + v * RM::LPR + gl);
    }
    float mx;
    const float w = a * row_softmax<KPAD>(m, gv, scale, p, mx);
    if (valid) {
#pragma unroll
      for (int v = 0; v < RM::VEC; ++v) {
        const int c = (v * RM::LPR + gl) * 4;
        float* dst = plan + row * k;
        if (c + 0 < k) dst[c + 0] = p[v].x * w;
        if (c + 1 < k) dst[c + 1] = p[v].y * w;
        if (c + 2 < k) dst[c + 2] = p[v].z * w;
        if (c + 3 < k) dst[c + 3] = p[v].w * w;
      }
    }
  }
}

template <typename T>
__global__ void assign_plan_kernel(const T* __restrict__ plan, long long n, int k, long long ld,
                                   int32_t* __restrict__ label) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const T* row = plan + i * ld;
  T best = row[0];
  int arg = 0;
  for (int j = 1; j < k; ++j) {
    const T v = row[j];
    if (v > best) { best = v; arg = j; }         // strict '>' keeps the first maximum (np.argmax)
  }
  label[i] = arg;
}

// label_i = argmax_j (g_j - M_ij), first max wins; centroid sums in shared memory.
// One warp per row (coalesced d-float read of X).  The accumulators [k][d] are replicated `copies` times;
// with one copy per warp (copies == warps) a warp owns its copy and adds without atomics, otherwise warps
// sharing a copy use shared-memory atomics.  Copies are folded into the fp64 global sums every flush_rows.
__global__ void __launch_bounds__(256)
assign_centroid_kernel(const float* __restrict__ M, long long n, int k, int kpad, const float* __restrict__ g,
                       const float* __restrict__ X, int d, int32_t* __restrict__ label, double* __restrict__ sum,
                       long long* __restrict__ cnt, int flush_rows, int copies) {
  extern __shared__ __align__(16) float acc_sh[];   // [copies][k*d], then cnt_sh [copies][k] (int)
  const int kd = k * d;
  int* cnt_sh = reinterpret_cast<int*>(acc_sh + (size_t)copies * kd);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, n_warps = blockDim.x >> 5;
  const bool exclusive = copies == n_warps;
  float* my_acc = acc_sh + (size_t)(warp % copies) * kd;
  int* my_cnt = cnt_sh + (warp % copies) * k;
  __shared__ float g_sh[256];
  for (int x = tid; x < k; x += blockDim.x) g_sh[x] = g ? g[x] : 0.f;
  for (int x = tid; x < copies * kd; x += blockDim.x) acc_sh[x] = 0.f;
  for (int x = tid; x < copies * k; x += blockDim.x) cnt_sh[x] = 0;
  __syncthreads();
  const long long per = (n + gridDim.x - 1) / gridDim.x;
  const long long r0 = per * blockIdx.x < n ? per * blockIdx.x : n;
  const long long r1 = r0 + per < n ? r0 + per : n;
  for (long long c0 = r0; c0 < r1; c0 += flush_rows) {
    const long long c1 = c0 + flush_rows < r1 ? c0 + flush_rows : r1;
    if (k <= 32) {
      // small k: a THREAD finds its row's label (k compares over its own kpad floats), then the warp walks
      // its 32 rows and adds each 4*d-byte row of X into the label's accumulator with coalesced loads
      for (long long row0 = c0 + (long long)warp * 32; row0 < c1; row0 += (long long)n_warps * 32) {
        const long long row = row0 + lane;
        const bool valid = row < c1;
        int arg = 0;
        if (valid && !M) arg = label[row];              // labels given: sums only
        if (valid && M) {
          float best = -INFINITY;
          const float4* mr = reinterpret_cast<const float4*>(M + row * kpad);
          for (int j4 = 0; j4 * 4 < k; ++j4) {
            const float4 m = __ldg(mr + j4);
            const float v[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int j = j4 * 4 + q;
              if (j < k) {
                const float t = g_sh[j] - v[q];
                if (t > best) { best = t; arg = j; }      // strict '>' keeps the first maximum
              }
            }
          }
          label[row] = arg;
        }
        const int n_valid = (int)((c1 - row0) < 32 ? (c1 - row0) : 32);
        for (int r = 0; r < n_valid; ++r) {
          const int lab = __shfl_sync(0xffffffffu, arg, r);
          if (lane == 0) { if (exclusive) my_cnt[lab] += 1; else atomicAdd(&my_cnt[lab], 1); }
          if (X) {
            const float* xr = X + (row0 + r) * d;
            float* ar = my_acc + (size_t)lab * d;
            if (exclusive) for (int t = lane; t < d; t += 32) ar[t] += __ldg(xr + t);
            else for (int t = lane; t < d; t += 32) atomicAdd(&ar[t], __ldg(xr + t));
          }
        }
      }
    } else
    for (long long row = c0 + warp; row < c1; row += n_warps) {
      float best = -INFINITY;
      int arg = 0x7fffffff;
      if (!M) {
        arg = label[row];                               // labels given: sums only
      } else {
        for (int j = lane; j < k; j += 32) {
          const float v = g_sh[j] - __ldg(M + row * kpad + j);
          if (v > best) { best = v; arg = j; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ob = __shfl_xor_sync(0xffffffffu, best, o);
          const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
          if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
        }
      }
      if (lane == 0) {
        if (M) label[row] = arg;
        if (exclusive) my_cnt[arg] += 1; else atomicAdd(&my_cnt[arg], 1);
      }
      if (X) {
        const float* xr = X + row * d;
        float* ar = my_acc + (size_t)arg * d;
        if (exclusive) for (int t = lane; t < d; t += 32) ar[t] += __ldg(xr + t);
        else for (int t = lane; t < d; t += 32) atomicAdd(&ar[t], __ldg(xr + t));
      }
    }
    __syncthreads();
    if (X)
      for (int x = tid; x < kd; x += blockDim.x) {
        float v = 0.f;
        for (int c = 0; c < copies; ++c) { v += acc_sh[(size_t)c * kd + x]; acc_sh[(size_t)c * kd + x] = 0.f; }
        if (v != 0.f) atomicAdd(sum + x, (double)v);
      }
    for (int x = tid; x < k; x += blockDim.x) {
      int v = 0;
      for (int c = 0; c < copies; ++c) { v += cnt_sh[c * k + x]; cnt_sh[c * k + x] = 0; }
      if (v) atomicAdd(reinterpret_cast<unsigned long long*>(cnt + x), (unsigned long long)v);
    }
    __syncthreads();
  }
}

// Small k (<= 32): the centroid sums stay in REGISTERS.  A lane finds the label of its own row, then the warp
// walks its 32 rows: the row of X is read coalesced (lane t holds columns t, t+32, ...), and since the label is
// warp-uniform the add goes to the accumulator registers of that label under a uniform predicate -- no shared-
// memory read-modify-write chain per row (the limiter of assign_centroid_kernel: 0.4 TB/s at n = 1 M).
// KT >= k accumulator sets of DT = ceil(d/32) floats per lane; folded over the CTA's warps in shared memory,
// then one fp64 atomic per (label, column) and CTA.
template <int KT, int DT>
__global__ void __launch_bounds__(256)
assign_centroid_reg_kernel(const float* __restrict__ M, long long n, int k, int kpad, const float* __restrict__ g,
                           const float* __restrict__ X, int d, int32_t* __restrict__ label, double* __restrict__ sum,
                           long long* __restrict__ cnt) {
  constexpr int NWARP = 8;
  __shared__ float g_sh[32];
  constexpr int FA = (KT * DT < 16) ? KT * DT : 16;   // accumulators folded per round (16 KB of shared memory)
  __shared__ float fold_sh[NWARP][FA * 32];
  __shared__ int cnt_sh[NWARP][32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < 32) g_sh[tid] = (tid < k && g) ? g[tid] : -INFINITY;
  __syncthreads();
  float acc[KT][DT];
#pragma unroll
  for (int j = 0; j < KT; ++j)
#pragma unroll
    for (int t = 0; t < DT; ++t) acc[j][t] = 0.f;
  int my_cnt = 0;                                     // rows with label == lane
  const long long per = (n + gridDim.x - 1) / gridDim.x;
  const long long r0 = per * blockIdx.x < n ? per * blockIdx.x : n;
  const long long r1 = r0 + per < n ? r0 + per : n;
  for (long long row0 = r0 + (long long)warp * 32; row0 < r1; row0 += (long long)NWARP * 32) {
    const long long row = row0 + lane;
    int arg = -1;
    if (row < r1 && !M) arg = label[row];               // labels given (balanced rounding ran): sums only
    if (row < r1 && M) {
      float best = -INFINITY;
      arg = 0;
      const float4* mr = reinterpret_cast<const float4*>(M + row * kpad);
      for (int j4 = 0; j4 * 4 < k; ++j4) {
        const float4 m = __ldg(mr + j4);
        const float v[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int j = j4 * 4 + q;
          const float t = g_sh[j & 31] - v[q];
          if (j < k && t > best) { best = t; arg = j; }       // strict '>' keeps the first maximum
        }
      }
      label[row] = arg;
    }
#pragma unroll
    for (int j = 0; j < KT; ++j) {
      const int c = __popc(__ballot_sync(0xffffffffu, arg == j));
      if (lane == j) my_cnt += c;
    }
    if (X) {
      const int n_valid = (int)((r1 - row0) < 32 ? (r1 - row0) : 32);
      for (int rb = 0; rb < n_valid; rb += 4) {             // 4 rows of X in flight
        float x[4][DT];
        int lab[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          lab[u] = __shfl_sync(0xffffffffu, arg, (rb + u) & 31);
          const bool ok = rb + u < n_valid;
          if (!ok) lab[u] = -1;
          const float* xr = X + (row0 + rb + (ok ? u : 0)) * d;
#pragma unroll
          for (int t = 0; t < DT; ++t) x[u][t] = (ok && lane + 32 * t < d) ? __ldg(xr + lane + 32 * t) : 0.f;
        }
        // acc[lab] += x as a mask-multiply over all labels: a predicated add would be turned into an indexed
        // (local-memory) access by the compiler
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int j = 0; j < KT; ++j) {
            const float mj = lab[u] == j ? 1.f : 0.f;
#pragma unroll
            for (int t = 0; t < DT; ++t) acc[j][t] = fmaf(mj, x[u][t], acc[j][t]);
          }
      }
    }
  }
  // fold the warps, FA accumulators per round
  cnt_sh[warp][lane] = my_cnt;
#pragma unroll
  for (int a0 = 0; a0 < KT * DT; a0 += FA) {
#pragma unroll
    for (int a = 0; a < FA; ++a) fold_sh[warp][a * 32 + lane] = acc[(a0 + a) / DT][(a0 + a) % DT];
    __syncthreads();
    if (X)
      for (int x = tid; x < FA * 32; x += blockDim.x) {
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < NWARP; ++w) v += fold_sh[w][x];
        const int ai = a0 + x / 32, j = ai / DT, col = (ai % DT) * 32 + (x & 31);
        if (j < k && col < d && v != 0.f) atomicAdd(sum + (size_t)j * d + col, (double)v);
      }
    __syncthreads();
  }
  if (tid < k) {
    int v = 0;
#pragma unroll
    for (int w = 0; w < NWARP; ++w) v += cnt_sh[w][tid];
    if (v) atomicAdd(reinterpret_cast<unsigned long long*>(cnt + tid), (unsigned long long)v);
  }
}

#define URE_KPAD_SWITCH(kpad, CALL)                    \
  switch (kpad) {                                      \
    case 8: { constexpr int KP = 8; CALL; } break;     \
    case 16: { constexpr int KP = 16; CALL; } break;   \
    case 32: { constexpr int KP = 32; CALL; } break;   \
    case 64: { constexpr int KP = 64; CALL; } break;   \
    case 128: { constexpr int KP = 128; CALL; } break; \
    case 256: { constexpr int KP = 256; CALL; } break; \
    default:                                           \
      set_error("kpad=%d not in {8,16,32,64,128,256}", kpad); \
      return URE_EUNSUPPORTED;                         \
  }

int check_mk(const void* M, long long n, int k, int kpad, const char* who) {
  URE_REQUIRE(M != nullptr, URE_EINVAL, "%s: null cost matrix", who);
  URE_REQUIRE(n > 0 && k >= 1 && k <= kpad, URE_EINVAL, "%s: bad shape n=%lld k=%d kpad=%d", who, n, k, kpad);
  return 0;
}

template <int KPAD>
int launch_sinkhorn(const float* M, long long n, int k, float* g, const SkStages& st, SkWorkspace* ws, int grid,
                    size_t smem, cudaStream_t stream) {
  auto kern = sinkhorn_kernel<KPAD>;
  URE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  URE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kSkThreads, smem));
  URE_REQUIRE(occ >= 1, URE_ECOOP, "sinkhorn_kernel<%d> cannot be resident (smem %zu)", KPAD, smem);
  void* args[] = {(void*)&M, (void*)&n, (void*)&k, (void*)&g, (void*)&st, (void*)&ws};
  URE_CUDA(cudaLaunchCooperativeKernel((void*)kern, dim3(grid), dim3(kSkThreads), args, smem, stream));
  return 0;
}

}  // namespace
}  // namespace ure

extern "C" int ure_sinkhorn_colsum(const float* d_M, int64_t n, int k, int kpad, const float* d_g, float eps,
                                   double n_total, double* d_colsum, void* stream) {
  using namespace ure;
  if (int rc = check_mk(d_M, n, k, kpad, "ure_sinkhorn_colsum")) return rc;
  URE_REQUIRE(d_g && d_colsum && eps > 0.f && n_total >= 1.0, URE_EINVAL, "ure_sinkhorn_colsum: bad argument");
  const float scale = kLog2e / eps;
  const double a = 1.0 / n_total;
  auto st = static_cast<cudaStream_t>(stream);
  // grid = one full wave of resident CTAs (a second, partly filled wave costs as much as a full one: 489 CTAs on
  // 444 slots ran at half speed), fewer only when there are not 512 rows per CTA
  auto grid_for = [&](const void* kern) -> unsigned {
    int occ = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kSkThreads, 0) != cudaSuccess || occ < 1) occ = 1;
    long long blocks = (n + 511) / 512;
    const long long cap = (long long)num_sms() * occ;
    if (blocks > cap) blocks = cap;
    return (unsigned)(blocks < 1 ? 1 : blocks);
  };
  if (k <= 8 && kpad != 8) {
    // only the first 8 columns hold centroids (the rest of the kpad-wide row is +inf padding): read that 32-byte
    // slice of every row -- half the exponentials at kpad = 16 (the bytes still come from DRAM in 64-byte pieces;
    // kernels.kpad_for stores such matrices 8 wide to begin with)
    colsum_kernel<8><<<grid_for((const void*)colsum_kernel<8>), kSkThreads, 0, st>>>(d_M, n, k, d_g, scale, a, d_colsum, kpad);
  } else {
    URE_KPAD_SWITCH(kpad, (colsum_kernel<KP><<<grid_for((const void*)colsum_kernel<KP>), kSkThreads, 0, st>>>(
                              d_M, n, k, d_g, scale, a, d_colsum, kpad)));
  }
  URE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int ure_sinkhorn_update_g(float* d_g, double* d_colsum, int k, float eps, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_g && d_colsum && k >= 1 && k <= 256 && eps > 0.f, URE_EINVAL, "ure_sinkhorn_update_g: bad argument");
  update_g_kernel<<<1, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_g, d_colsum, k, eps);
  URE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int64_t ure_sinkhorn_workspace_bytes(void) { return (int64_t)sizeof(ure::SkWorkspace); }

extern "C" int ure_sinkhorn(const float* d_M, int64_t n, int k, int kpad, float* d_g, const float* h_eps,
                            const int32_t* h_iters, int n_stages, float tol, void* d_workspace, void* stream) {
  using namespace ure;
  if (int rc = check_mk(d_M, n, k, kpad, "ure_sinkhorn")) return rc;
  URE_REQUIRE(d_g && h_eps && h_iters && d_workspace, URE_EINVAL, "ure_sinkhorn: null argument");
  URE_REQUIRE(n_stages >= 1 && n_stages <= kMaxStages, URE_EINVAL, "ure_sinkhorn: n_stages=%d outside [1,%d]",
              n_stages, kMaxStages);
  SkStages stg;
  stg.n = n_stages;
  stg.tol = tol;
  for (int s = 0; s < n_stages; ++s) {
    URE_REQUIRE(h_eps[s] > 0.f && h_iters[s] >= 0, URE_EINVAL, "ure_sinkhorn: stage %d eps/iters invalid", s);
    stg.eps[s] = h_eps[s];
    stg.iters[s] = h_iters[s];
  }
  auto st = static_cast<cudaStream_t>(stream);
  auto* ws = static_cast<SkWorkspace*>(d_workspace);
  URE_CUDA(cudaMemsetAsync(ws, 0, sizeof(SkWorkspace), st));
  const int grid = num_sms();
  const long long per = (n + grid - 1) / grid;
  const size_t parts = 2 * (size_t)(kSkThreads / 32) * kpad * sizeof(float);   // per-warp (r, s) column partials
  const size_t need = (size_t)per * kpad * sizeof(float) + parts;
  if (kpad <= 64) {
    // tiny problem: one thread-block cluster, M in its CTAs' shared memory, column sums exchanged through
    // distributed shared memory, a hardware cluster barrier per iteration
    const long long per_c = (n + kClusterMax - 1) / kClusterMax;
    const int ks = k <= 8 ? 8 : kpad;                // columns kept in shared memory
    const size_t need_c = (size_t)per_c * ks * sizeof(float);
    if (need_c <= 160 * 1024) {
      // (only kpad <= 64 reaches this point: the static shared memory of the wider instantiations would not fit)
#define URE_CLUSTER_CASE(KP)                                                                                      \
  if (kpad == KP)                                                                                                 \
    return ks == 8 ? launch_sinkhorn_cluster<KP, 8>(d_M, n, k, d_g, stg, ws, kClusterMax, need_c, st)             \
                   : launch_sinkhorn_cluster<KP, KP>(d_M, n, k, d_g, stg, ws, kClusterMax, need_c, st);
      URE_CLUSTER_CASE(8) URE_CLUSTER_CASE(16) URE_CLUSTER_CASE(32) URE_CLUSTER_CASE(64)
#undef URE_CLUSTER_CASE
    }
  }
  int smem_optin = 0;
  {
    int dev = 0;
    URE_CUDA(cudaGetDevice(&dev));
    URE_CUDA(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  }
  if ((long long)need <= (long long)smem_optin - 2048) {     // minus the kernel's static shared memory
    // the cost rows fit the SMs' shared memory (n = 1 M users at k <= 8: 216 KB per SM): one persistent launch, M is
    // read from HBM once for ALL iterations, an iteration costs a shared-memory sweep + one grid barrier
    URE_KPAD_SWITCH(kpad, return (launch_sinkhorn<KP>(d_M, n, k, d_g, stg, ws, grid, need, st)));
  }
  // large problem: one streaming pass per iteration at full occupancy (split-phase kernels, no host sync;
  // the early exit needs the column sums on the host, so every scheduled iteration runs)
  for (int s = 0; s < n_stages; ++s)
    for (int it = 0; it < h_iters[s]; ++it) {
      if (int rc = ure_sinkhorn_colsum(d_M, n, k, kpad, d_g, h_eps[s], (double)n, ws->colsum[0], stream)) return rc;
      if (int rc = ure_sinkhorn_update_g(d_g, ws->colsum[0], k, h_eps[s], stream)) return rc;
    }
  return 0;
}

extern "C" int64_t ure_sinkhorn_peer_xchg_bytes(void) { return (int64_t)sizeof(ure::SkXchg); }

extern "C" int ure_sinkhorn_peer(const float* d_M, int64_t n_local, double n_total, int k, int kpad, float* d_g,
                                 const float* h_eps, const int32_t* h_iters, int n_stages, float tol,
                                 const uint64_t* h_xchg_ptrs, int rank, int world, uint64_t call_base,
                                 void* d_workspace, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_M && d_g && h_eps && h_iters && h_xchg_ptrs && d_workspace, URE_EINVAL, "ure_sinkhorn_peer: null argument");
  URE_REQUIRE(n_local >= 0 && n_total >= 1.0 && k >= 1 && k <= kpad && kpad <= 256, URE_EINVAL,
              "ure_sinkhorn_peer: bad shape n_local=%lld k=%d kpad=%d", (long long)n_local, k, kpad);
  URE_REQUIRE(world >= 1 && world <= kPeerMax && rank >= 0 && rank < world, URE_EINVAL,
              "ure_sinkhorn_peer: rank %d of %d (at most %d GPUs)", rank, world, kPeerMax);
  URE_REQUIRE(n_stages >= 1 && n_stages <= kMaxStages, URE_EINVAL, "ure_sinkhorn_peer: n_stages=%d", n_stages);
  SkStages stg;
  stg.n = n_stages;
  stg.tol = tol;
  for (int s = 0; s < n_stages; ++s) {
    URE_REQUIRE(h_eps[s] > 0.f && h_iters[s] >= 0, URE_EINVAL, "ure_sinkhorn_peer: stage %d eps/iters invalid", s);
    stg.eps[s] = h_eps[s];
    stg.iters[s] = h_iters[s];
  }
  SkPeers peers;
  for (int r = 0; r < kPeerMax; ++r) peers.xchg[r] = reinterpret_cast<unsigned long long*>(r < world ? h_xchg_ptrs[r] : 0);
  auto st = static_cast<cudaStream_t>(stream);
  auto* ws = static_cast<SkWorkspace*>(d_workspace);
  URE_CUDA(cudaMemsetAsync(ws, 0, sizeof(SkWorkspace), st));
  long long nn = n_local;
  unsigned long long base = call_base;
  int stride = kpad;
  void* args[] = {(void*)&d_M, (void*)&nn, (void*)&n_total, (void*)&k, (void*)&d_g, (void*)&stg, (void*)&ws,
                  (void*)&peers, (void*)&rank, (void*)&world, (void*)&base, (void*)&stride};
  // every CTA the GPU can keep resident (cooperative launch), fewer only when there are not 512 rows per CTA
  auto launch = [&](const void* kern) -> int {
    int occ = 1;
    URE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kSkThreads, 0));
    URE_REQUIRE(occ >= 1, URE_ECOOP, "sinkhorn_peer_kernel cannot be resident");
    long long grid = (n_local + 511) / 512;
    if (grid > (long long)num_sms() * occ) grid = (long long)num_sms() * occ;
    if (grid < 1) grid = 1;
    URE_CUDA(cudaLaunchCooperativeKernel(kern, dim3((unsigned)grid), dim3(kSkThreads), args, 0, st));
    return 0;
  };
  if (k <= 8 && kpad != 8) return launch((const void*)sinkhorn_peer_kernel<8>);     // the 8-column slice of every row
  URE_KPAD_SWITCH(kpad, return launch((const void*)sinkhorn_peer_kernel<KP>));
  return 0;
}

extern "C" int ure_sinkhorn_plan(const float* d_M, int64_t n, int k, int kpad, const float* d_g, float eps,
                                 double n_total, float* d_plan, void* stream) {
  using namespace ure;
  if (int rc = check_mk(d_M, n, k, kpad, "ure_sinkhorn_plan")) return rc;
  URE_REQUIRE(d_g && d_plan && eps > 0.f && n_total >= 1.0, URE_EINVAL, "ure_sinkhorn_plan: bad argument");
  const float scale = kLog2e / eps, a = (float)(1.0 / n_total);
  long long blocks = (n + 255) / 256;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  auto st = static_cast<cudaStream_t>(stream);
  URE_KPAD_SWITCH(kpad, (plan_kernel<KP><<<(unsigned)blocks, 256, 0, st>>>(d_M, n, k, d_g, scale, a, d_plan)));
  URE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int ure_assign_plan_f64(const double* d_plan, int64_t n, int k, int64_t ld, int32_t* d_label,
                                   void* stream) {
  using namespace ure;
  URE_REQUIRE(d_plan && d_label && n > 0 && k >= 1 && ld >= k, URE_EINVAL, "ure_assign_plan_f64: bad argument");
  assign_plan_kernel<double><<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      d_plan, n, k, ld, d_label);
  URE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int ure_assign_plan_f32(const float* d_plan, int64_t n, int k, int64_t ld, int32_t* d_label,
                                   void* stream) {
  using namespace ure;
  URE_REQUIRE(d_plan && d_label && n > 0 && k >= 1 && ld >= k, URE_EINVAL, "ure_assign_plan_f32: bad argument");
  assign_plan_kernel<float><<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      d_plan, n, k, ld, d_label);
  URE_CUDA(cudaGetLastError());
  return 0;
}

namespace ure {
// d_M == NULL: the labels are an input (after the balanced rounding) and only the sums / counts are computed
static int assign_centroids_impl(const float* d_M, int64_t n, int k, int kpad, const float* d_g,
                                 const float* d_X, int d, int32_t* d_label, double* d_sum, int64_t* d_cnt,
                                 void* stream) {
  const int dd = d_X ? d : 0;
  {
    // register path: k <= 32 and at most 64 accumulators per lane
    const int kt = k <= 8 ? 8 : k <= 16 ? 16 : k <= 32 ? 32 : 0;
    const int dt = dd <= 32 ? 1 : dd <= 64 ? 2 : dd <= 128 ? 4 : 0;
    if (kt && dt && kt * dt <= 64) {
      long long blocks = (n + 2047) / 2048;
      const long long cap = (long long)num_sms() * 2;       // one wave of resident CTAs: the fp64 atomics of the
      if (blocks > cap) blocks = cap;                         // final fold (k*d addresses) scale with the CTA count
      auto st = static_cast<cudaStream_t>(stream);
      auto* cntp = reinterpret_cast<long long*>(d_cnt);
#define URE_ASSIGN_REG(KT_, DT_)                                                                              \
  if (kt == KT_ && dt == DT_) {                                                                             \
    assign_centroid_reg_kernel<KT_, DT_><<<(unsigned)blocks, 256, 0, st>>>(d_M, n, k, kpad, d_g, d_X, dd, d_label, \
                                                                          d_sum, cntp);                      \
    URE_CUDA(cudaGetLastError());                                                                            \
    return 0;                                                                                                \
  }
      URE_ASSIGN_REG(8, 1) URE_ASSIGN_REG(8, 2) URE_ASSIGN_REG(8, 4) URE_ASSIGN_REG(16, 1) URE_ASSIGN_REG(16, 2)
      URE_ASSIGN_REG(16, 4) URE_ASSIGN_REG(32, 1) URE_ASSIGN_REG(32, 2)
#undef URE_ASSIGN_REG
    }
  }
  const size_t one = ((size_t)k * dd + k) * sizeof(float);
  URE_REQUIRE(one <= 200 * 1024, URE_EUNSUPPORTED, "ure_assign_centroids: k*d=%d too large for shared memory", k * d);
  int copies = (int)((96 * 1024) / one);            // <= 96 KB: two CTAs per SM stay resident
  if (copies > 8) copies = 8;                        // 8 warps per CTA
  if (copies < 1) copies = 1;
  while (copies > 1 && (8 % copies) != 0) --copies;  // warps map evenly onto copies
  const size_t smem = one * copies;
  URE_CUDA(cudaFuncSetAttribute(assign_centroid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  long long blocks = (n + 1023) / 1024;
  const long long cap = (long long)num_sms() * 2;
  if (blocks > cap) blocks = cap;
  assign_centroid_kernel<<<(unsigned)blocks, 256, smem, static_cast<cudaStream_t>(stream)>>>(
      d_M, n, k, kpad, d_g, d_X, dd, d_label, d_sum, reinterpret_cast<long long*>(d_cnt), 4096, copies);
  URE_CUDA(cudaGetLastError());
  return 0;
}
}  // namespace ure

extern "C" int ure_assign_centroids(const float* d_M, int64_t n, int k, int kpad, const float* d_g,
                                    const float* d_X, int d, int32_t* d_label, double* d_sum, int64_t* d_cnt,
                                    void* stream) {
  using namespace ure;
  if (int rc = check_mk(d_M, n, k, kpad, "ure_assign_centroids")) return rc;
  URE_REQUIRE(d_g && d_label && d_cnt && (!d_X || (d_sum && d > 0)), URE_EINVAL, "ure_assign_centroids: bad argument");
  return assign_centroids_impl(d_M, n, k, kpad, d_g, d_X, d, d_label, d_sum, d_cnt, stream);
}

extern "C" int ure_centroid_sums(const float* d_X, int64_t n, int d, const int32_t* d_label, int k, double* d_sum,
                                 int64_t* d_cnt, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_X && d_label && d_sum && d_cnt && n > 0 && d > 0 && k >= 1 && k <= 256, URE_EINVAL,
              "ure_centroid_sums: bad argument");
  return assign_centroids_impl(nullptr, n, k, 16, nullptr, d_X, d, const_cast<int32_t*>(d_label), d_sum, d_cnt, stream);
}
