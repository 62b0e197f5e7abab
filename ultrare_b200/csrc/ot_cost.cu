// User-to-centroid squared-euclidean cost matrix on the 5th-gen tensor cores.
//
// Replaces  dist = ((X - centroid[:, None])**2).sum(axis=2)   (reference
// method/utils.py:637, a NumPy broadcast that materialises [k,n,d]) by
//     M[i,j] = ||x_i||^2 + ||c_j||^2 - 2 * (X C^T)[i,j]
// with the contraction X C^T issued as tcgen05.mma kind::tf32 on 128-row tiles and
// fp32 accumulators in TMEM.  Plain TF32 (10-bit mantissa) would destroy the 1e-5
// relative cost tolerance the Sinkhorn plan needs (SURVEY.md H5), so both operands
// are split x = hi + lo with hi = x & 0xFFFFE000 (exactly representable in tf32) and
// three MMAs hi*hi + hi*lo + lo*hi are accumulated: error ~2^-21 relative.
//
// Pipeline per CTA (persistent over row tiles, 128 threads):
//   bulk-TMA (cp.async.bulk, 1-D) stages the raw fp32 tile [128, d] into shared memory
//   under an mbarrier; all threads split it into the K-major no-swizzle UMMA core-matrix
//   layout ([d/4 chunks][128 rows][16 B]) and reduce the row norms; one thread issues
//   3*d/8 MMAs and commits to an mbarrier; the four warps read their 32 TMEM lanes back
//   with tcgen05.ld, apply the norm epilogue and store the rows of M.
// The problem is bound by reading X (4*n*d bytes), not by the tensor pipe (Appendix D).
#include <cuda.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace ure {
namespace {

constexpr int kCostThreads = 512;      // 16 warps: transform + epilogue are instruction bound with fewer

struct CostSmemLayout {
  uint32_t raw_off, raw_stage_bytes, stages;
  uint32_t a_hi, a_lo, lbo_a;
  uint32_t b_hi, b_lo, lbo_b;
  uint32_t xnorm, rowmin, cnorm, bars, holder, total;
};

__host__ __device__ inline CostSmemLayout cost_layout(int D, int NB, int stages) {
  CostSmemLayout L;
  const uint32_t chunks = D / 4;
  L.lbo_a = kTileRows * 16 + (chunks >= 8 ? 16 : 32);
  L.lbo_b = NB * 16 + (chunks >= 8 ? 16 : 32);
  uint32_t o = 0;
  L.stages = stages;
  L.raw_stage_bytes = kTileRows * D * 4;
  L.raw_off = o; o += L.raw_stage_bytes * stages;
  L.a_hi = o; o += L.lbo_a * chunks;
  L.a_lo = o; o += L.lbo_a * chunks;
  L.b_hi = o; o += L.lbo_b * chunks;
  L.b_lo = o; o += L.lbo_b * chunks;
  L.xnorm = o; o += kTileRows * 4;
  L.rowmin = o; o += kTileRows * 4;
  L.cnorm = o; o += NB * 4;
  L.bars = o; o += 8 * 4;       // full[2], mma
  L.holder = o; o += 16;
  L.total = o;
  return L;
}

template <int D>
__global__ void __launch_bounds__(kCostThreads)
cost_tc_kernel(const float* __restrict__ X, long long n, const float* __restrict__ C, int k, int kpad, int NB,
               int stages, uint32_t tmem_cols, float* __restrict__ M, double* __restrict__ inertia) {
  constexpr int CH = D / 4;                    // 16-byte K chunks per row
  extern __shared__ __align__(128) unsigned char sm[];
  const CostSmemLayout L = cost_layout(D, NB, stages);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint64_t* full = reinterpret_cast<uint64_t*>(sm + L.bars);
  uint64_t* mma_bar = full + 2;
  uint32_t* holder = reinterpret_cast<uint32_t*>(sm + L.holder);
  float* xnorm = reinterpret_cast<float*>(sm + L.xnorm);
  int* rowmin = reinterpret_cast<int*>(sm + L.rowmin);     // float bits (costs are >= 0: int order == float order)
  float* cnorm = reinterpret_cast<float*>(sm + L.cnorm);
  const int col0 = blockIdx.y * NB;            // first centroid column of this CTA

  if (tid == 0) {
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    mbar_init(mma_bar, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(holder, tmem_cols);

  // ---- centroid block -> B_hi / B_lo (K-major core-matrix layout) + ||c||^2
  for (int idx = tid; idx < NB * CH; idx += kCostThreads) {
    const int j = idx / CH, c = idx % CH;
    const int col = col0 + j;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (col < k) v = __ldg(reinterpret_cast<const float4*>(C + (size_t)col * D) + c);
    float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
    float4 lo = make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
    *reinterpret_cast<float4*>(sm + L.b_hi + c * L.lbo_b + j * 16) = hi;
    *reinterpret_cast<float4*>(sm + L.b_lo + c * L.lbo_b + j * 16) = lo;
    float s = (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
#pragma unroll
    for (int o = CH / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, CH);
    if (c == 0) cnorm[j] = col < k ? s : INFINITY;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *holder;
  const uint32_t idesc = make_idesc_tf32(NB);
  const uint32_t a_hi_addr = smem_u32(sm + L.a_hi), a_lo_addr = smem_u32(sm + L.a_lo);
  const uint32_t b_hi_addr = smem_u32(sm + L.b_hi), b_lo_addr = smem_u32(sm + L.b_lo);

  const long long n_tiles = (n + kTileRows - 1) / kTileRows;
  auto tile_bytes = [&](long long tile) -> uint32_t {
    const long long rows = (n - tile * kTileRows) < kTileRows ? (n - tile * kTileRows) : kTileRows;
    return (uint32_t)(rows * D * 4);
  };
  auto issue_load = [&](long long tile, int stage) {
    const uint32_t bytes = tile_bytes(tile);
    mbar_expect_tx(&full[stage], bytes);
    bulk_g2s(sm + L.raw_off + (size_t)stage * L.raw_stage_bytes, X + tile * kTileRows * (long long)D, bytes, &full[stage]);
  };

  long long tile = blockIdx.x;
  if (tid == 0 && tile < n_tiles) issue_load(tile, 0);
  double inertia_acc = 0.0;
  for (int it = 0; tile < n_tiles; ++it, tile += gridDim.x) {
    const int stage = stages == 2 ? (it & 1) : 0;
    const uint32_t full_parity = stages == 2 ? ((it >> 1) & 1) : (it & 1);
    const long long next = tile + gridDim.x;
    if (stages == 2 && tid == 0 && next < n_tiles) issue_load(next, stage ^ 1);
    mbar_wait(&full[stage], full_parity);

    // ---- split the raw tile into hi / lo operand tiles, reduce row norms
    const float* raw = reinterpret_cast<const float*>(sm + L.raw_off + (size_t)stage * L.raw_stage_bytes);
    if (tid < kTileRows) rowmin[tid] = 0x7f800000;          // +inf
#pragma unroll 4
    for (int idx = tid; idx < kTileRows * CH; idx += kCostThreads) {
      const int r = idx / CH, c = idx % CH;
      const float4 v = *reinterpret_cast<const float4*>(raw + r * D + c * 4);
      const float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
      const float4 lo = make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
      *reinterpret_cast<float4*>(sm + L.a_hi + c * L.lbo_a + r * 16) = hi;
      *reinterpret_cast<float4*>(sm + L.a_lo + c * L.lbo_a + r * 16) = lo;
      float s = (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
#pragma unroll
      for (int o = CH / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, CH);
      if (c == 0) xnorm[r] = s;
    }
    fence_proxy_async();          // generic-proxy smem writes -> visible to the tensor-core (async) proxy
    __syncthreads();

    if (tid == 0) {
      if (stages == 1 && next < n_tiles) issue_load(next, 0);     // raw tile fully consumed
      tc_fence_after();
#pragma unroll
      for (int kk = 0; kk < D / 8; ++kk) {
        const uint64_t ah = make_desc(a_hi_addr + kk * 2 * L.lbo_a, L.lbo_a, 128);
        const uint64_t al = make_desc(a_lo_addr + kk * 2 * L.lbo_a, L.lbo_a, 128);
        const uint64_t bh = make_desc(b_hi_addr + kk * 2 * L.lbo_b, L.lbo_b, 128);
        const uint64_t bl = make_desc(b_lo_addr + kk * 2 * L.lbo_b, L.lbo_b, 128);
        umma_tf32(tmem_base, ah, bh, idesc, kk > 0);
        umma_tf32(tmem_base, ah, bl, idesc, 1);
        umma_tf32(tmem_base, al, bh, idesc, 1);
      }
      umma_commit(mma_bar);       // implies tcgen05.fence::before_thread_sync
    }
    mbar_wait(mma_bar, it & 1);
    tc_fence_after();

    // ---- epilogue: warp w reads TMEM lanes 32*(w%4).. (its row quarter) and every 4th 16-column chunk
    const int rq = warp & 3, cg = warp >> 2;
    const int trow = rq * 32 + lane;
    const long long row = tile * kTileRows + trow;
    const float xn = xnorm[trow];
    float rmin = INFINITY;
    for (int c0 = cg * 16; c0 < NB; c0 += 16 * (kCostThreads / 128)) {
      float acc[16];
      tmem_ld16(tmem_base + ((uint32_t)(rq * 32) << 16) + (uint32_t)c0, acc);
      if (row < n) {
        float out[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          out[j] = fmaf(-2.f, acc[j], xn + cnorm[c0 + j]);
          rmin = fminf(rmin, out[j]);
        }
        float4* dst = reinterpret_cast<float4*>(M + row * kpad + col0 + c0);
#pragma unroll
        for (int q = 0; q < 4; ++q)            // kpad == 8: the 16-column accumulator block is stored as 32-byte rows
          if (4 * q < kpad) dst[q] = make_float4(out[4 * q], out[4 * q + 1], out[4 * q + 2], out[4 * q + 3]);
      }
    }
    if (inertia && row < n && rmin < INFINITY) atomicMin(&rowmin[trow], __float_as_int(fmaxf(rmin, 0.f)));
    tc_fence_before();
    __syncthreads();              // TMEM accumulator and A tiles may be overwritten now
    if (inertia && tid < kTileRows && tile * kTileRows + tid < n) inertia_acc += (double)__int_as_float(rowmin[tid]);
    __syncthreads();              // rowmin is re-initialised by the next tile
  }
  if (inertia) {
    inertia_acc = warp_sum(inertia_acc);
    if (lane == 0 && inertia_acc != 0.0) atomicAdd(inertia, inertia_acc);
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, tmem_cols);
}

// ------------------------------------------------------------------ v2: tensor-map TMA straight into the UMMA layout
// Measured on the B200 (v1 handed the UNTRUNCATED tile as its hi operand: same results): tcgen05 kind::tf32 ignores the
// low 13 mantissa bits of its operands, so the RAW fp32 tile is a valid `hi` operand: hi*B is computed on the truncated values either way.  The
// tile therefore goes from global memory directly into the K-major core-matrix layout the tensor core reads
// ([d/4 chunks][128 rows][16 B]: one 2-D TMA box {4 floats, 128 rows} per chunk, cp.async.bulk.tensor), and the only
// generic-proxy pass left is lo = x - trunc(x) plus the row norms: half the shared-memory stores of v1, none of its
// bank conflicts (threads walk rows, 16 contiguous bytes each), and a footprint that lets two CTAs share an SM at
// d = 64 so that one CTA's TMA / MMA / epilogue latencies are covered by the other's work.
struct CostSmemLayout2 {
  uint32_t hi_off, stage_bytes, stages, lo_off, lbo_a;
  uint32_t b_hi, b_lo, lbo_b;
  uint32_t xnorm, rowmin, cnorm, bars, holder, total;
};

__host__ __device__ inline CostSmemLayout2 cost_layout2(int D, int NB, int stages) {
  CostSmemLayout2 L;
  const uint32_t chunks = D / 4;
  L.lbo_a = kTileRows * 16;                   // (no swizzle) a TMA box lands as 128 contiguous 16-byte rows
  L.lbo_b = NB * 16 + (chunks >= 8 ? 16 : 32);
  uint32_t o = 0;
  L.stages = stages;
  L.stage_bytes = kTileRows * D * 4;
  L.hi_off = o; o += L.stage_bytes * stages;
  L.lo_off = o; o += L.stage_bytes;
  L.b_hi = o; o += L.lbo_b * chunks;
  L.b_lo = o; o += L.lbo_b * chunks;
  L.xnorm = o; o += kTileRows * 4;
  L.rowmin = o; o += kTileRows * 4;
  L.cnorm = o; o += NB * 4;
  o = (o + 7) / 8 * 8;
  L.bars = o; o += 8 * 4;                     // full[2], mma
  L.holder = o; o += 16;
  L.total = o;
  return L;
}

// SW: the tile is loaded as D/32 boxes of {32 floats = 128 bytes, 128 rows} with the 128-byte swizzle (one wide box
// per 16 KB instead of eight 16-byte-wide ones: the TMA engine moves whole 128-byte rows) and the A descriptors say
// SWIZZLE_128B; lo is written at the SAME offsets as the raw tile, so the pass needs no index arithmetic at all.
template <int D, bool SW>
__global__ void __launch_bounds__(kCostThreads)
cost_tma_kernel(const __grid_constant__ CUtensorMap tmap, long long n, const float* __restrict__ C, int k, int kpad, int NB,
                int stages, uint32_t tmem_cols, float* __restrict__ M, double* __restrict__ inertia, int nacc) {
  constexpr int CH = D / 4;                    // 16-byte K chunks per row
  extern __shared__ __align__(128) unsigned char sm_raw[];
  // the swizzle atoms want 1024-byte aligned tiles: the launch asks for 1 KB more than the layout
  unsigned char* const sm = sm_raw + ((1024u - (smem_u32(sm_raw) & 1023u)) & 1023u);
  const CostSmemLayout2 L = cost_layout2(D, NB, stages);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint64_t* full = reinterpret_cast<uint64_t*>(sm + L.bars);
  uint64_t* mma_bar = full + 2;
  uint32_t* holder = reinterpret_cast<uint32_t*>(sm + L.holder);
  float* xnorm = reinterpret_cast<float*>(sm + L.xnorm);
  int* rowmin = reinterpret_cast<int*>(sm + L.rowmin);     // float bits (costs are >= 0: int order == float order)
  float* cnorm = reinterpret_cast<float*>(sm + L.cnorm);
  const int col0 = blockIdx.y * NB;            // first centroid column of this CTA

  if (tid == 0) {
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    mbar_init(mma_bar, 1);
    fence_mbar_init();
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
  }
  if (warp == 0) tmem_alloc(holder, tmem_cols);

  // ---- centroid block -> B_hi / B_lo (K-major core-matrix layout) + ||c||^2
  for (int idx = tid; idx < NB * CH; idx += kCostThreads) {
    const int j = idx / CH, c = idx % CH;
    const int col = col0 + j;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (col < k) v = __ldg(reinterpret_cast<const float4*>(C + (size_t)col * D) + c);
    float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
    float4 lo = make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
    *reinterpret_cast<float4*>(sm + L.b_hi + c * L.lbo_b + j * 16) = hi;
    *reinterpret_cast<float4*>(sm + L.b_lo + c * L.lbo_b + j * 16) = lo;
    float s = (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
#pragma unroll
    for (int o = CH / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, CH);
    if (c == 0) cnorm[j] = col < k ? s : INFINITY;
  }
  if (tid < kTileRows) xnorm[tid] = 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *holder;
  const uint32_t idesc = make_idesc_tf32(NB);
  const uint32_t a_lo_addr = smem_u32(sm + L.lo_off);
  const uint32_t b_hi_addr = smem_u32(sm + L.b_hi), b_lo_addr = smem_u32(sm + L.b_lo);

  const long long n_tiles = (n + kTileRows - 1) / kTileRows;
  auto issue_load = [&](long long tile, int stage) {          // CH boxes of {4 floats, 128 rows}: rows past n are zeros
    mbar_expect_tx(&full[stage], L.stage_bytes);
    unsigned char* dst = sm + L.hi_off + (size_t)stage * L.stage_bytes;
    if (SW) {
#pragma unroll
      for (int a = 0; a < D / 32; ++a) tma_load_2d(dst + a * (kTileRows * 128), &tmap, 32 * a, (int)(tile * kTileRows), &full[stage]);
    } else {
#pragma unroll 4
      for (int c = 0; c < CH; ++c) tma_load_2d(dst + c * L.lbo_a, &tmap, 4 * c, (int)(tile * kTileRows), &full[stage]);
    }
  };

  long long tile = blockIdx.x;
  if (tid == 0 && tile < n_tiles) issue_load(tile, 0);
  double inertia_acc = 0.0;
  for (int it = 0; tile < n_tiles; ++it, tile += gridDim.x) {
    const int stage = stages == 2 ? (it & 1) : 0;
    const uint32_t full_parity = stages == 2 ? ((it >> 1) & 1) : (it & 1);
    const long long next = tile + gridDim.x;
    if (stages == 2 && tid == 0 && next < n_tiles) issue_load(next, stage ^ 1);
    mbar_wait(&full[stage], full_parity);

    // ---- lo = x - trunc(x) in the same layout, row norms; threads walk rows (16 contiguous bytes each)
    const unsigned char* hi = sm + L.hi_off + (size_t)stage * L.stage_bytes;
    if (tid < kTileRows) rowmin[tid] = 0x7f800000;          // +inf
    if (SW) {
      // linear walk over the tile's 16-byte chunks: 8 consecutive chunks are one 128-byte row of one K atom
#pragma unroll 4
      for (int x = tid; x < kTileRows * CH; x += kCostThreads) {
        const float4 v = *reinterpret_cast<const float4*>(hi + x * 16);
        const float4 lo = make_float4(v.x - tf32_hi(v.x), v.y - tf32_hi(v.y), v.z - tf32_hi(v.z), v.w - tf32_hi(v.w));
        *reinterpret_cast<float4*>(sm + L.lo_off + x * 16) = lo;
        float s = (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        s += __shfl_xor_sync(0xffffffffu, s, 4);
        if ((tid & 7) == 0) atomicAdd(&xnorm[(x >> 3) & (kTileRows - 1)], s);
      }
    } else {
      const int r = tid & (kTileRows - 1), cg = tid / kTileRows;
      float s = 0.f;
#pragma unroll 4
      for (int c = cg; c < CH; c += kCostThreads / kTileRows) {
        const float4 v = *reinterpret_cast<const float4*>(hi + c * L.lbo_a + r * 16);
        const float4 lo = make_float4(v.x - tf32_hi(v.x), v.y - tf32_hi(v.y), v.z - tf32_hi(v.z), v.w - tf32_hi(v.w));
        *reinterpret_cast<float4*>(sm + L.lo_off + c * L.lbo_a + r * 16) = lo;
        s += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
      }
      if (cg < CH) atomicAdd(&xnorm[r], s);
    }
    fence_proxy_async();          // generic-proxy smem writes -> visible to the tensor-core (async) proxy
    __syncthreads();

    if (tid == 0) {
      tc_fence_after();
      const uint32_t a_hi_addr = smem_u32(hi);
#pragma unroll
      for (int kk = 0; kk < D / 8; ++kk) {
        // SW: K atom kk / 4 (16 KB each), 32 bytes further inside the atom per instruction
        const uint32_t a_off = SW ? (uint32_t)((kk >> 2) * (kTileRows * 128) + (kk & 3) * 32) : (uint32_t)(kk * 2 * L.lbo_a);
        const uint64_t ah = SW ? make_desc_sw128(a_hi_addr + a_off) : make_desc(a_hi_addr + a_off, L.lbo_a, 128);
        const uint64_t al = SW ? make_desc_sw128(a_lo_addr + a_off) : make_desc(a_lo_addr + a_off, L.lbo_a, 128);
        const uint64_t bh = make_desc(b_hi_addr + kk * 2 * L.lbo_b, L.lbo_b, 128);
        const uint64_t bl = make_desc(b_lo_addr + kk * 2 * L.lbo_b, L.lbo_b, 128);
        // nacc == 3: hi*hi, hi*lo and lo*hi accumulate in three TMEM column blocks -- three independent chains of
        // D/8 instructions instead of one chain of 3*D/8 whose every link waits for the previous accumulator update
        umma_tf32(tmem_base, ah, bh, idesc, kk > 0);       // the tensor core truncates the raw tile to tf32 itself
        umma_tf32(tmem_base + (nacc == 3 ? NB : 0), ah, bl, idesc, nacc == 3 ? kk > 0 : 1);
        umma_tf32(tmem_base + (nacc == 3 ? 2 * NB : 0), al, bh, idesc, nacc == 3 ? kk > 0 : 1);
      }
      umma_commit(mma_bar);       // implies tcgen05.fence::before_thread_sync
    }
    mbar_wait(mma_bar, it & 1);
    tc_fence_after();
    if (stages == 1 && tid == 0 && next < n_tiles) issue_load(next, 0);     // the MMAs have consumed the raw tile

    // ---- epilogue: warp w reads TMEM lanes 32*(w%4).. (its row quarter) and every 4th 16-column chunk
    const int rq = warp & 3, cg = warp >> 2;
    const int trow = rq * 32 + lane;
    const long long row = tile * kTileRows + trow;
    const float xn = xnorm[trow];
    float rmin = INFINITY;
    for (int c0 = cg * 16; c0 < NB; c0 += 16 * (kCostThreads / 128)) {
      float acc[16];
      tmem_ld16(tmem_base + ((uint32_t)(rq * 32) << 16) + (uint32_t)c0, acc);
      if (nacc == 3) {
        float a2[16];
        tmem_ld16(tmem_base + ((uint32_t)(rq * 32) << 16) + (uint32_t)(NB + c0), a2);
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[j] += a2[j];
        tmem_ld16(tmem_base + ((uint32_t)(rq * 32) << 16) + (uint32_t)(2 * NB + c0), a2);
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[j] += a2[j];
      }
      if (row < n) {
        float out[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          out[j] = fmaf(-2.f, acc[j], xn + cnorm[c0 + j]);
          rmin = fminf(rmin, out[j]);
        }
        float4* dst = reinterpret_cast<float4*>(M + row * kpad + col0 + c0);
#pragma unroll
        for (int q = 0; q < 4; ++q)            // kpad == 8: the 16-column accumulator block is stored as 32-byte rows
          if (4 * q < kpad) dst[q] = make_float4(out[4 * q], out[4 * q + 1], out[4 * q + 2], out[4 * q + 3]);
      }
    }
    if (inertia && row < n && rmin < INFINITY) atomicMin(&rowmin[trow], __float_as_int(fmaxf(rmin, 0.f)));
    tc_fence_before();
    __syncthreads();              // TMEM accumulator, the lo tile and xnorm may be overwritten now
    if (tid < kTileRows) {
      if (inertia && tile * kTileRows + tid < n) inertia_acc += (double)__int_as_float(rowmin[tid]);
      xnorm[tid] = 0.f;
    }
    __syncthreads();              // rowmin / xnorm are re-initialised before the next tile's passes
  }
  if (inertia) {
    inertia_acc = warp_sum(inertia_acc);
    if (lane == 0 && inertia_acc != 0.0) atomicAdd(inertia, inertia_acc);
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, tmem_cols);
}

// *used = 1 when the TMA kernel was launched (2: the caller still owes the inertia pass), 0 when the caller should
// use v1 (no driver entry point / odd shape); the return value is an error code as everywhere
template <int D>
int launch_cost_tma(const float* X, long long n, const float* C, int k, int kpad, float* M, double* inertia, cudaStream_t st,
                    int* used) {
  *used = 0;
  EncodeTiledFn enc = encode_tiled();
  if (!enc || D < 8 || (reinterpret_cast<uintptr_t>(X) & 15) != 0 || n >= (1ll << 31)) return 0;
  // column block and stages: prefer a footprint that lets two CTAs share an SM
  const int kcols = kpad < 16 ? 16 : kpad;      // kpad == 8: a 16-column MMA block, 8 columns stored
  int NB = kcols > 128 ? 128 : kcols, stages = 2;
  while (kcols % NB) NB -= 16;
  if (cost_layout2(D, NB, 2).total > 109 * 1024 && cost_layout2(D, NB, 1).total <= 109 * 1024) stages = 1;
  if (cost_layout2(D, NB, stages).total > 219 * 1024) stages = 1;
  if (cost_layout2(D, NB, stages).total > 219 * 1024) return 0;
  const int col_blocks = kcols / NB;
  const int nacc = 3 * NB <= 256 ? 3 : 1;      // two CTAs per SM share the 512 TMEM columns
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < nacc * NB) tmem_cols <<= 1;
  constexpr bool sw = D >= 32;                 // a 128-byte swizzle atom is 32 floats of K
  CUtensorMap tmap;
  const cuuint64_t dims[2] = {(cuuint64_t)D, (cuuint64_t)n};
  const cuuint64_t strides[1] = {(cuuint64_t)D * 4};
  const cuuint32_t box[2] = {sw ? 32u : 4u, (cuuint32_t)kTileRows};
  const cuuint32_t estr[2] = {1, 1};
  if (enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(X), dims, strides, box, estr,
          CU_TENSOR_MAP_INTERLEAVE_NONE, sw ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
          CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return 0;
  const CostSmemLayout2 L = cost_layout2(D, NB, stages);
  auto kern = cost_tma_kernel<D, sw>;
  const size_t smem = (size_t)L.total + 1024;
  URE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  URE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  int occ = 0;
  URE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kCostThreads, smem));
  if (occ < 1) return 0;
  const int max_by_tmem = 512 / (int)tmem_cols;
  if (occ > max_by_tmem) occ = max_by_tmem;
  if (occ > 4) occ = 4;
  *used = 1;
  const long long n_tiles = (n + kTileRows - 1) / kTileRows;
  long long gx = (long long)num_sms() * occ / col_blocks;
  if (gx < 1) gx = 1;
  if (gx > n_tiles) gx = n_tiles;
  double* fused_inertia = (col_blocks == 1) ? inertia : nullptr;
  kern<<<dim3((unsigned)gx, (unsigned)col_blocks), kCostThreads, smem, st>>>(tmap, n, C, k, kpad, NB, stages, tmem_cols, M,
                                                                         fused_inertia, nacc);
  URE_CUDA(cudaGetLastError());
  if (inertia && !fused_inertia) *used = 2;
  return 0;
}

// ------------------------------------------------------------------ v4: warp-specialised pipeline (d >= 32, kpad <= 64)
// ncu of the kernels above (profiles/r2_notes.md): a CTA walks  TMA wait -> lo pass -> MMAs -> commit wait -> epilogue
// strictly one after the other -- 28 % of the stall samples sit on the MMA-completion mbarrier alone (with N = 16 every
// instruction re-reads a 4 KB A slab from shared memory for 16 columns of output), the rest on the TMA and the
// barriers in between.  Here every stage has its own warps and the stages of consecutive tiles overlap:
//   warp 0      TMA producer: S raw tiles in flight (128-byte-swizzled boxes, the raw tile IS the hi operand);
//   warps 1-8   lo = x - trunc(x) into one of two lo tiles, row norms (8 slots deep);
//   warp 9      MMA issuer: D1 [128 x 2NB] += A_hi x [B_hi ; B_lo]^T  (hi*hi and hi*lo in ONE instruction: the A slab
//               is read once for both), D2 [128 x NB] += A_lo x B_hi^T; two accumulator stages in TMEM; three
//               tcgen05.commit release the raw tile, the lo tile and publish the accumulators;
//   warps 10-13 epilogue: tcgen05.ld of D1[:, :NB] + D1[:, NB:] + D2, norms, rows of M, inertia.
constexpr int kWsThreads = 14 * 32;
constexpr int kWsLoWarps = 8;

struct CostWsLayout {
  uint32_t hi_off, tile_bytes, S, lo_off, LS, b_off, lbo_b, xnorm, cnorm, bars, holder, total;
};
__host__ __device__ inline CostWsLayout cost_ws_layout(int D, int NB) {
  CostWsLayout L;
  const uint32_t chunks = D / 4;
  L.tile_bytes = kTileRows * D * 4;
  L.lbo_b = 2 * NB * 16 + (chunks >= 8 ? 16 : 32);      // [B_hi ; B_lo]: 2 NB rows per 16-byte K chunk
  // raw (hi) and lo tile stages: as many as fit next to the centroid block (226 KB per CTA)
  const uint32_t fixed = L.lbo_b * chunks + 8 * kTileRows * 4 + NB * 4 + 16 * 8 + 16 + 64 + 1024;
  const uint32_t tiles = fixed < 226u * 1024u ? (226u * 1024u - fixed) / L.tile_bytes : 0u;
  L.S = tiles >= 6 ? 4 : tiles >= 4 ? 3 : 2;
  L.LS = tiles >= 5 ? 2 : 1;
  if (tiles < 3) L.S = 0;                                // does not fit: the caller falls back
  uint32_t o = 0;
  L.hi_off = o; o += L.tile_bytes * L.S;
  L.lo_off = o; o += L.tile_bytes * L.LS;
  L.b_off = o; o += L.lbo_b * chunks;
  L.xnorm = o; o += 8 * kTileRows * 4;
  L.cnorm = o; o += NB * 4;
  o = (o + 7) / 8 * 8;
  L.bars = o; o += 16 * 8;                               // full[4] empty[4] lo_full[2] lo_empty[2] t_full[2] t_empty[2]
  L.holder = o; o += 16;
  L.total = o;
  return L;
}

template <int D>
__global__ void __launch_bounds__(kWsThreads, 1)
cost_ws_kernel(const __grid_constant__ CUtensorMap tmap, long long n, const float* __restrict__ C, int k, int kpad, int NB,
               uint32_t tmem_cols, int fold, float* __restrict__ M, double* __restrict__ inertia) {
  constexpr int CH = D / 4;
  extern __shared__ __align__(128) unsigned char sm_raw[];
  unsigned char* const sm = sm_raw + ((1024u - (smem_u32(sm_raw) & 1023u)) & 1023u);
  const CostWsLayout L = cost_ws_layout(D, NB);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint64_t* const full = reinterpret_cast<uint64_t*>(sm + L.bars);
  uint64_t* const empty = full + 4;
  uint64_t* const lo_full = full + 8;
  uint64_t* const lo_empty = full + 10;
  uint64_t* const t_full = full + 12;
  uint64_t* const t_empty = full + 14;
  uint32_t* const holder = reinterpret_cast<uint32_t*>(sm + L.holder);
  float* const xnorm = reinterpret_cast<float*>(sm + L.xnorm);        // [8][128]
  float* const cnorm = reinterpret_cast<float*>(sm + L.cnorm);
  const int S = (int)L.S, LS = (int)L.LS;

  if (tid == 0) {
    for (int i = 0; i < 4; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&lo_full[i], kWsLoWarps * 32); mbar_init(&lo_empty[i], 1);
      mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], 128);
    }
    fence_mbar_init();
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
  }
  if (warp == 0) tmem_alloc(holder, tmem_cols);
  // ---- centroids -> [B_hi ; B_lo] (K-major core-matrix layout, no swizzle) + ||c||^2
  for (int idx = tid; idx < NB * CH; idx += kWsThreads) {
    const int j = idx / CH, c = idx % CH;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (j < k) v = __ldg(reinterpret_cast<const float4*>(C + (size_t)j * D) + c);
    const float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
    const float4 lo = make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
    *reinterpret_cast<float4*>(sm + L.b_off + c * L.lbo_b + j * 16) = hi;
    *reinterpret_cast<float4*>(sm + L.b_off + c * L.lbo_b + (NB + j) * 16) = lo;
    float s = (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
#pragma unroll
    for (int o = CH / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, CH);
    if (c == 0) cnorm[j] = j < k ? s : INFINITY;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *holder;
  const long long n_tiles = (n + kTileRows - 1) / kTileRows;
  const int my_tiles = blockIdx.x < n_tiles ? (int)((n_tiles - 1 - blockIdx.x) / gridDim.x) + 1 : 0;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0)
      for (int it = 0; it < my_tiles; ++it) {
        const int s = it % S;
        const long long tile = blockIdx.x + (long long)it * gridDim.x;
        mbar_wait(&empty[s], (uint32_t)(((it / S) & 1) ^ 1));
        mbar_expect_tx(&full[s], L.tile_bytes);
        unsigned char* dst = sm + L.hi_off + (size_t)s * L.tile_bytes;
#pragma unroll
        for (int a = 0; a < D / 32; ++a) tma_load_2d(dst + a * (kTileRows * 128), &tmap, 32 * a, (int)(tile * kTileRows), &full[s]);
      }
  } else if (warp <= kWsLoWarps) {
    // ------------------------------------------------------------ lo pass + row norms
    // Thread = (row, half of the row's eight 16-byte positions in every 128-byte atom row): the norm of a row is a
    // private sum + ONE shuffle (no shared-memory atomics: a float atomicAdd there is a compare-and-swap loop), and
    // lo lands at the address its hi came from, so the swizzle never has to be undone.  Position j of the four is
    // rotated by the row number: the 8 threads of a quarter-warp (4 rows x 2 halves) hit 8 different bank groups.
    const int lt = tid - 32;                                    // 0 .. 255
    const int lrow = lt >> 1, lhalf = lt & 1;
    uint32_t pos[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) pos[j] = (uint32_t)(lrow * 128 + (lhalf * 4 + ((j + lrow) & 3)) * 16);
    for (int it = 0; it < my_tiles; ++it) {
      const int s = it % S, ls = it % LS;
      mbar_wait(&full[s], (uint32_t)((it / S) & 1));
      mbar_wait(&lo_empty[ls], (uint32_t)(((it / LS) & 1) ^ 1));
      const unsigned char* hi = sm + L.hi_off + (size_t)s * L.tile_bytes;
      unsigned char* lo = sm + L.lo_off + (size_t)ls * L.tile_bytes;
      float4 v[D / 32][4];
#pragma unroll
      for (int a = 0; a < D / 32; ++a)
#pragma unroll
        for (int j = 0; j < 4; ++j) v[a][j] = *reinterpret_cast<const float4*>(hi + a * (kTileRows * 128) + pos[j]);
      float q0 = 0.f, q1 = 0.f;
#pragma unroll
      for (int a = 0; a < D / 32; ++a)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 x = v[a][j];
          *reinterpret_cast<float4*>(lo + a * (kTileRows * 128) + pos[j]) =
              make_float4(x.x - tf32_hi(x.x), x.y - tf32_hi(x.y), x.z - tf32_hi(x.z), x.w - tf32_hi(x.w));
          q0 = fmaf(x.x, x.x, fmaf(x.y, x.y, q0));
          q1 = fmaf(x.z, x.z, fmaf(x.w, x.w, q1));
        }
      float q = q0 + q1;
      q += __shfl_xor_sync(0xffffffffu, q, 1);
      if (lhalf == 0) xnorm[(it & 7) * kTileRows + lrow] = q;   // slot read by the epilogue, reused eight tiles later
      fence_proxy_async();                                      // lo is read by the tensor core (async proxy)
      mbar_arrive(&lo_full[ls]);
    }
  } else if (warp == kWsLoWarps + 1) {
    // ------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      const uint32_t idesc2 = make_idesc_tf32(2 * NB), idesc1 = make_idesc_tf32(NB);
      const uint32_t b_addr = smem_u32(sm + L.b_off);
      for (int it = 0; it < my_tiles; ++it) {
        const int s = it % S, ls = it % LS, a = it & 1;
        mbar_wait(&lo_full[ls], (uint32_t)((it / LS) & 1));
        mbar_wait(&t_empty[a], (uint32_t)(((it >> 1) & 1) ^ 1));
        tc_fence_after();
        const uint32_t hi_addr = smem_u32(sm + L.hi_off + (size_t)s * L.tile_bytes);
        const uint32_t lo_addr = smem_u32(sm + L.lo_off + (size_t)ls * L.tile_bytes);
        if (!fold) {
          const uint32_t d1 = tmem_base + (uint32_t)(a * 3 * NB), d2 = d1 + (uint32_t)(2 * NB);
#pragma unroll
          for (int kk = 0; kk < D / 8; ++kk) {
            const uint32_t a_off = (uint32_t)((kk >> 2) * (kTileRows * 128) + (kk & 3) * 32);
            const uint64_t bdesc = make_desc(b_addr + kk * 2 * L.lbo_b, L.lbo_b, 128);
            umma_tf32(d1, make_desc_sw128(hi_addr + a_off), bdesc, idesc2, kk > 0);     // hi*hi | hi*lo
            umma_tf32(d2, make_desc_sw128(lo_addr + a_off), bdesc, idesc1, kk > 0);     // lo*hi (first NB rows of B)
          }
        } else {
          // wide centroid blocks (6 NB columns of TMEM do not exist): the three products go to ONE accumulator
          const uint32_t dd = tmem_base + (uint32_t)(a * NB);
#pragma unroll
          for (int kk = 0; kk < D / 8; ++kk) {
            const uint32_t a_off = (uint32_t)((kk >> 2) * (kTileRows * 128) + (kk & 3) * 32);
            const uint64_t bhi = make_desc(b_addr + kk * 2 * L.lbo_b, L.lbo_b, 128);
            const uint64_t blo = make_desc(b_addr + kk * 2 * L.lbo_b + (uint32_t)NB * 16u, L.lbo_b, 128);
            const uint64_t ahi = make_desc_sw128(hi_addr + a_off);
            umma_tf32(dd, ahi, bhi, idesc1, kk > 0);
            umma_tf32(dd, ahi, blo, idesc1, 1);
            umma_tf32(dd, make_desc_sw128(lo_addr + a_off), bhi, idesc1, 1);
          }
        }
        umma_commit(&empty[s]);             // the raw tile may be overwritten by the producer
        umma_commit(&lo_empty[ls]);         // ... the lo tile by the lo warps
        umma_commit(&t_full[a]);            // ... and the accumulators are complete
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue: one TMEM lane = one row per thread
    const int rq = warp & 3;
    const int trow = rq * 32 + lane;
    double inertia_acc = 0.0;
    for (int it = 0; it < my_tiles; ++it) {
      const int a = it & 1;
      const long long tile = blockIdx.x + (long long)it * gridDim.x;
      const long long row = tile * kTileRows + trow;
      mbar_wait(&t_full[a], (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      float* xn = xnorm + (it & 7) * kTileRows;
      const float xnr = xn[trow];
      const uint32_t d1 = tmem_base + ((uint32_t)(rq * 32) << 16) + (uint32_t)(a * (fold ? 1 : 3) * NB);
      float rmin = INFINITY;
      for (int c0 = 0; c0 < NB; c0 += 16) {
        float acc[16], t2[16];
        tmem_ld16(d1 + (uint32_t)c0, acc);
        if (!fold) {
          tmem_ld16(d1 + (uint32_t)(NB + c0), t2);
#pragma unroll
          for (int j = 0; j < 16; ++j) acc[j] += t2[j];
          tmem_ld16(d1 + (uint32_t)(2 * NB + c0), t2);
#pragma unroll
          for (int j = 0; j < 16; ++j) acc[j] += t2[j];
        }
        if (row < n) {
          float out[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            out[j] = fmaf(-2.f, acc[j], xnr + cnorm[c0 + j]);
            rmin = fminf(rmin, out[j]);
          }
          float4* dst = reinterpret_cast<float4*>(M + row * kpad + c0);
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (c0 + 4 * q < kpad) dst[q] = make_float4(out[4 * q], out[4 * q + 1], out[4 * q + 2], out[4 * q + 3]);
        }
      }
      tc_fence_before();
      mbar_arrive(&t_empty[a]);
      if (inertia && row < n && rmin < INFINITY) inertia_acc += (double)fmaxf(rmin, 0.f);
    }
    if (inertia) {
      inertia_acc = warp_sum(inertia_acc);
      if (lane == 0 && inertia_acc != 0.0) atomicAdd(inertia, inertia_acc);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, tmem_cols);
}

// *used = 1 when the pipeline kernel ran
template <int D>
int launch_cost_ws(const float* X, long long n, const float* C, int k, int kpad, float* M, double* inertia, cudaStream_t st,
                   int* used) {
  *used = 0;
  EncodeTiledFn enc = encode_tiled();
  const int NB = kpad < 16 ? 16 : kpad;
  if (!enc || D < 32 || NB > 128 || (reinterpret_cast<uintptr_t>(X) & 15) != 0 || n >= (1ll << 31)) return 0;
  const CostWsLayout L = cost_ws_layout(D, NB);
  const size_t smem = (size_t)L.total + 1024;
  if (L.S == 0 || smem > 227 * 1024) return 0;
  const int fold = 6 * NB > 512;                              // TMEM has 512 columns
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < (fold ? 2 : 6) * NB) tmem_cols <<= 1;   // two accumulator stages of [D1 (2 NB) | D2 (NB)], or of one [NB]
  CUtensorMap tmap;
  const cuuint64_t dims[2] = {(cuuint64_t)D, (cuuint64_t)n};
  const cuuint64_t strides[1] = {(cuuint64_t)D * 4};
  const cuuint32_t box[2] = {32u, (cuuint32_t)kTileRows};
  const cuuint32_t estr[2] = {1, 1};
  if (enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(X), dims, strides, box, estr,
          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return 0;
  auto kern = cost_ws_kernel<D>;
  URE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long n_tiles = (n + kTileRows - 1) / kTileRows;
  long long gx = num_sms();
  if (gx > n_tiles) gx = n_tiles;
  *used = 1;
  kern<<<dim3((unsigned)gx), kWsThreads, smem, st>>>(tmap, n, C, k, kpad, NB, tmem_cols, fold, M, inertia);
  URE_CUDA(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ CUDA-core check kernel
// Direct fp32 sum_t (x-c)^2 (the reference expression): one thread per (row, column).
__global__ void cost_simt_kernel(const float* __restrict__ X, long long n, int d, const float* __restrict__ C, int k,
                                 int kpad, float* __restrict__ M) {
  const long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= n * kpad) return;
  const long long i = x / kpad;
  const int j = (int)(x % kpad);
  float s = INFINITY;
  if (j < k) {
    s = 0.f;
    for (int t = 0; t < d; ++t) {
      const float df = __ldg(X + i * d + t) - __ldg(C + (size_t)j * d + t);
      s = fmaf(df, df, s);
    }
  }
  M[x] = s;
}

__global__ void rowmin_sum_kernel(const float* __restrict__ M, long long n, int k, int kpad, double* __restrict__ out) {
  double acc = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float m = INFINITY;
    for (int j = 0; j < k; ++j) m = fminf(m, M[i * kpad + j]);
    acc += (double)m;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0 && acc != 0.0) atomicAdd(out, acc);
}

int launch_rowmin(const float* M, long long n, int k, int kpad, double* inertia, cudaStream_t st) {
  long long blocks = (n + 255) / 256;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  rowmin_sum_kernel<<<(unsigned)blocks, 256, 0, st>>>(M, n, k, kpad, inertia);
  URE_CUDA(cudaGetLastError());
  return 0;
}

template <int D>
int launch_cost_tc(const float* X, long long n, const float* C, int k, int kpad, float* M, double* inertia,
                   cudaStream_t st) {
  if constexpr (D >= 32) {
    int used = 0;
    if (int rc = launch_cost_ws<D>(X, n, C, k, kpad, M, inertia, st, &used)) return rc;
    if (used) return 0;
  }
  {
    int used = 0;
    if (int rc = launch_cost_tma<D>(X, n, C, k, kpad, M, inertia, st, &used)) return rc;
    if (used == 1) return 0;
    if (used == 2) return launch_rowmin(M, n, k, kpad, inertia, st);
  }
  // choose the column block NB (multiple of 16) and the number of raw stages that fit in shared memory
  const uint32_t budget = 220 * 1024;
  const int kcols = kpad < 16 ? 16 : kpad;      // kpad == 8: a 16-column MMA block, 8 columns stored
  int NB = kcols, stages = 2;
  while (true) {
    if (cost_layout(D, NB, stages).total <= budget) break;
    if (stages == 2 && cost_layout(D, NB, 1).total <= budget) { stages = 1; break; }
    if (NB <= 16) { set_error("ure_cost_matrix: d=%d does not fit shared memory", D); return URE_EUNSUPPORTED; }
    NB = ((NB / 2 + 15) / 16) * 16;
    stages = 2;
  }
  const int col_blocks = (kcols + NB - 1) / NB;
  URE_REQUIRE(col_blocks * NB == kcols, URE_EUNSUPPORTED, "ure_cost_matrix: kpad=%d not divisible into %d-column blocks",
              kpad, NB);
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < NB) tmem_cols <<= 1;
  const CostSmemLayout L = cost_layout(D, NB, stages);
  auto kern = cost_tc_kernel<D>;
  URE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
  int occ = 0;
  URE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kCostThreads, L.total));
  URE_REQUIRE(occ >= 1, URE_EUNSUPPORTED, "ure_cost_matrix: kernel cannot be resident (smem %u)", L.total);
  const int max_by_tmem = 512 / (int)tmem_cols;
  if (occ > max_by_tmem) occ = max_by_tmem;
  if (occ > 8) occ = 8;
  const long long n_tiles = (n + kTileRows - 1) / kTileRows;
  long long gx = (long long)num_sms() * occ / col_blocks;
  if (gx < 1) gx = 1;
  if (gx > n_tiles) gx = n_tiles;
  double* fused_inertia = (col_blocks == 1) ? inertia : nullptr;
  kern<<<dim3((unsigned)gx, (unsigned)col_blocks), kCostThreads, L.total, st>>>(X, n, C, k, kpad, NB, stages, tmem_cols, M,
                                                                            fused_inertia);
  URE_CUDA(cudaGetLastError());
  if (inertia && !fused_inertia) return launch_rowmin(M, n, k, kpad, inertia, st);
  return 0;
}

int check_cost_args(const float* X, long long n, int d, const float* C, int k, int kpad, float* M, const char* who) {
  URE_REQUIRE(X && C && M, URE_EINVAL, "%s: null argument", who);
  URE_REQUIRE(n > 0 && k >= 1 && k <= kpad && (kpad == 8 || kpad % 16 == 0) && kpad <= 256, URE_EINVAL,
              "%s: bad shape n=%lld k=%d kpad=%d (kpad 8 or a multiple of 16, <= 256)", who, n, k, kpad);
  URE_REQUIRE(d >= 1, URE_EINVAL, "%s: d=%d", who, d);
  return 0;
}

}  // namespace
}  // namespace ure

extern "C" int ure_cost_matrix(const float* d_X, int64_t n, int d, const float* d_C, int k, int kpad, float* d_M,
                               double* d_inertia, void* stream) {
  using namespace ure;
  if (int rc = check_cost_args(d_X, n, d, d_C, k, kpad, d_M, "ure_cost_matrix")) return rc;
  auto st = static_cast<cudaStream_t>(stream);
  switch (d) {
    case 8: return launch_cost_tc<8>(d_X, n, d_C, k, kpad, d_M, d_inertia, st);
    case 16: return launch_cost_tc<16>(d_X, n, d_C, k, kpad, d_M, d_inertia, st);
    case 32: return launch_cost_tc<32>(d_X, n, d_C, k, kpad, d_M, d_inertia, st);
    case 64: return launch_cost_tc<64>(d_X, n, d_C, k, kpad, d_M, d_inertia, st);
    case 128: return launch_cost_tc<128>(d_X, n, d_C, k, kpad, d_M, d_inertia, st);
    default:
      set_error("ure_cost_matrix: d=%d not in {8,16,32,64,128}", d);
      return URE_EUNSUPPORTED;
  }
}

extern "C" int ure_cost_matrix_simt(const float* d_X, int64_t n, int d, const float* d_C, int k, int kpad,
                                    float* d_M, double* d_inertia, void* stream) {
  using namespace ure;
  if (int rc = check_cost_args(d_X, n, d, d_C, k, kpad, d_M, "ure_cost_matrix_simt")) return rc;
  auto st = static_cast<cudaStream_t>(stream);
  const long long total = n * kpad;
  cost_simt_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_X, n, d, d_C, k, kpad, d_M);
  URE_CUDA(cudaGetLastError());
  if (d_inertia) return launch_rowmin(d_M, n, k, kpad, d_inertia, st);
  return 0;
}
