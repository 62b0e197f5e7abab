// Owner-computes schedule of the fused MF training step (ure_mf_hparams_t::mode == URE_MF_OWNER).
//
// Same arithmetic as mf_train.cu (baseTrain, reference method/utils.py:58-98, + the dense
// optim.SGD(momentum, weight_decay) update of scratch.py:65-68), different data movement:
//
//   * Every CTA serves ONE shard and owns a contiguous slice of that shard's user rows and a slice of
//     its item rows.  The owned weights and momentum buffers live in shared memory for the whole launch.
//   * The shard's records exist twice, sorted by user and sorted by item (ure_mf_owner_prepare), so the
//     interactions of an owned row are one contiguous run of slots.  A batch is a random subset of the
//     shard (the per-epoch visiting order); which batch a slot belongs to in epoch e is
//     step_of(slot) = inverse_permutation_e(record index) / batch.  ure_mf_owner_schedule evaluates it for a
//     window of epochs in an embarrassingly parallel pre-pass and leaves, for every CTA, epoch and step, the
//     SORTED list of the CTA's slots in that batch (16-bit slot numbers in L2 / HBM): the training loop only
//     copies its next list into shared memory in the shadow of the barrier.
//   * A step walks the list in waves -- a group of d/4 lanes per interaction: the OTHER table's row is
//     gathered with 16-byte loads, the error is re-computed on both sides, the contributions of consecutive
//     interactions of the same row are summed in registers (in the group, then across the warp's groups by
//     a segmented shuffle reduction) and the run totals go to the row's shared-memory gradient; then every
//     owned row gets its SGD update in shared memory and its new weights are published.
//     No global atomics, no global gradient arrays, no separate dense sweep over HBM/L2.
//   * When they fit, the slots' (other index, rating, own row) are cached in shared memory as well, so the
//     only L2 traffic of a step is the gather of the other table's rows.
//   * Updated rows are published to the buffer the NEXT step reads: P/Q and gP/gQ alternate
//     (reads of step j come from buffer j&1), so gradients always see pre-step weights (batch-synchronous
//     semantics of the reference) with ONE barrier per step -- and only among the CTAs of the shard.
#include "common.cuh"
#include "feistel.cuh"
#include <string.h>
#include <type_traits>
#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace ure {
namespace {

constexpr int kOwnThreads = 512;
constexpr int KMAX = URE_MAX_SHARDS;

struct OwnerWs {
  int max_rows;           // written by plan_kernel: max owned rows (user + item) of a CTA
  int max_slots;          // max owned interactions (user side + item side) of a CTA
  int max_spe;            // max steps per epoch of a shard
  int avail_smem;         // dynamic shared memory a launch can get
  int error;              // set by the training kernel: 1 = a step outside the scheduled window was requested
  int pad0;
  int trace_steps;        // diagnostics (ure_mf_train_trace): stamps of the first trace_steps steps of a launch
  int pad1;
  long long* trace;       // [trace_steps][grid][6] SM-clock stamps, or NULL
  long long tot_slots;    // written by plan_kernel: sum over the shards of 2 n (slots of one schedule row)
  int pad[20];
  unsigned bar[KMAX][32]; // one barrier counter per shard, one 128-byte line each
  unsigned unsorted[KMAX]; // set by csr_count_kernel: the shard's records are NOT already in user-row order (zero on entry)
};

struct Plan {
  int shard, q, c;        // my shard, my index among its c CTAs
  int ru0, ru1, ri0, ri1; // owned user rows / item rows
  int su0, mU, si0, mI;   // first slot and slot count in inter_u / inter_i
  long long slot_base;    // first of the CTA's slots in a schedule row: 2 n of the shards before + su0 + si0
};

// first r in [0, n_rows] with off[r] >= target, moved down by one when that boundary is nearer
__device__ int nearest_boundary(const int32_t* off, int n_rows, long long target) {
  int lo = 0, hi = n_rows;                       // off[n_rows] = n >= target
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if ((long long)off[mid] >= target) hi = mid; else lo = mid + 1;
  }
  if (lo > 0 && target - (long long)off[lo - 1] < (long long)off[lo] - target) --lo;
  return lo;
}

// CTA -> (shard, row slices).  CTAs are apportioned to shards by interaction count (largest remainder);
// inside a shard CTA q takes user rows up to the boundary nearest q*n/c, and item rows so that the
// CUMULATIVE (user + item) slot count of CTAs 0..q-1 is nearest 2*q*n/c (items are the finer grain).
// The item slices are handed out either in row order or from the last row down, whichever gives the smaller
// maximum of owned rows per CTA: when row number and activity are correlated in both tables (ids sorted by
// popularity), pairing the many-row slice of one table with the few-row slice of the other is what lets the
// owned rows fit shared memory.
// Block-cooperative (any block size >= 32, ends with a __syncthreads); scratch in shared memory.
struct PlanScratch {
  int c[KMAX];
  long long rem[KMAX];
  int ub[KMAX + 1], ib[KMAX + 1], jb[KMAX + 1];
};

__device__ void make_plan(const ure_mf_shard_t* shards, int K, int cta, int n_cta, Plan& pl, PlanScratch& ps) {
  if (threadIdx.x == 0) {
    long long N = 0;
    for (int s = 0; s < K; ++s) N += shards[s].n;
    if (N < 1) N = 1;
    const long long spare = n_cta - K;
    int used = 0;
    for (int s = 0; s < K; ++s) {
      const long long x = spare * (long long)shards[s].n;
      ps.c[s] = 1 + (int)(x / N);
      ps.rem[s] = x % N;
      used += ps.c[s];
    }
    for (int left = n_cta - used; left > 0; --left) {
      int best = 0;
      for (int s = 1; s < K; ++s)
        if (ps.rem[s] > ps.rem[best]) best = s;
      ++ps.c[best];
      ps.rem[best] = -1;
    }
    int s = 0, base = 0;
    while (s < K - 1 && cta >= base + ps.c[s]) base += ps.c[s++];
    pl.shard = s; pl.q = cta - base; pl.c = ps.c[s];
    long long sb = 0;
    for (int x = 0; x < s; ++x) sb += 2ll * shards[x].n;
    pl.slot_base = sb;
  }
  __syncthreads();
  const ure_mf_shard_t& sh = shards[pl.shard];
  const int c = pl.c;
  const long long n = sh.n;
  // every boundary of the shard, in parallel; the item boundaries are made monotone by a running maximum
  for (int q = threadIdx.x; q <= c; q += blockDim.x) {
    int u = q <= 0 ? 0 : q >= c ? (int)sh.n_user : nearest_boundary(sh.off_u, sh.n_user, q * n / c);
    ps.ub[q] = u;
    const long long want = q <= 0 || q >= c ? 0 : 2 * q * n / c - (long long)sh.off_u[u];   // item slots of CTAs < q
    ps.ib[q] = q <= 0 ? 0 : q >= c ? (int)sh.n_item : nearest_boundary(sh.off_i, sh.n_item, want);
    ps.jb[q] = q <= 0 ? (int)sh.n_item : q >= c ? 0 : nearest_boundary(sh.off_i, sh.n_item, max(0ll, n - want));
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int up = 0, down = (int)sh.n_item, max_f = 0, max_r = 0;
    for (int q = 0; q <= c; ++q) {         // monotone boundaries; the owned-row maxima of both hand-out orders
      const int pu = up, pd = down;
      up = max(up, ps.ib[q]);
      down = min(down, ps.jb[q]);
      ps.ib[q] = up;
      ps.jb[q] = down;
      if (q > 0) {
        const int ru = ps.ub[q] - ps.ub[q - 1];
        max_f = max(max_f, ru + up - pu);
        max_r = max(max_r, ru + pd - down);
      }
    }
    const bool rev = max_r < max_f;
    pl.ru0 = ps.ub[pl.q]; pl.ru1 = ps.ub[pl.q + 1];
    pl.ri0 = rev ? ps.jb[pl.q + 1] : ps.ib[pl.q];
    pl.ri1 = rev ? ps.jb[pl.q] : ps.ib[pl.q + 1];
    pl.su0 = sh.off_u[pl.ru0]; pl.mU = sh.off_u[pl.ru1] - pl.su0;
    pl.si0 = sh.off_i[pl.ri0]; pl.mI = sh.off_i[pl.ri1] - pl.si0;
    // the CTA's slots in a schedule row start after those of the shard's CTAs before it
    pl.slot_base += (long long)pl.su0 + (rev ? n - (long long)sh.off_i[pl.ri1] : (long long)pl.si0);
  }
  __syncthreads();
}

// hparams.owner_plan (the workspace): the launch was queued with capacities from an earlier plan.  Every CTA of the
// schedule pre-pass compares them with the plan it derives; one that is not covered flags the workspace and does
// nothing else (block-uniform).  The training kernel starts after the pre-pass and trains nothing when the flag is up.
__device__ __forceinline__ bool plan_not_covered(const ure_mf_hparams_t& hp, const Plan& pl, int spe) {
  if (!hp.owner_plan) return false;
  const bool bad = (pl.ru1 - pl.ru0) + (pl.ri1 - pl.ri0) > hp.owner_cap_rows || pl.mU + pl.mI > hp.owner_cap_slots ||
                   spe > hp.owner_spe_cap;
  if (bad && threadIdx.x == 0) static_cast<OwnerWs*>(hp.owner_plan)->error = 2;
  return bad;
}

constexpr int kOtherBits = 20;            // record cache: other-table row in the low 20 bits, own row above
constexpr int kOwnWarps = kOwnThreads / 32;
constexpr int kMaxSpe = 8192;             // steps per epoch the schedule pre-pass handles (histogram in shared memory)

// Dynamic shared memory of the training kernel.  The layout depends on LAUNCH-uniform capacities only
// (cap_rows, cap_slots: the plan's maxima over the CTAs), so every array base is a uniform value:
//   boundary rows [2*warps][d] fp32 | batch list [cap_list] u16 | packed records 8 B: of every owned slot
//   [cap_slots] (record cache) or of the staged batch list [cap_list] | owned rows [cap_rows][2d] fp32 (w | momentum) | first / last boundary record of every row 2 x [cap_rows] int
__host__ __device__ inline long long owner_smem_bytes(int d, int cap_rows, int cap_slots, int cap_list, bool cached) {
  return 2ll * kOwnWarps * d * 4 + 2ll * cap_list + 8ll * (cached ? cap_slots : cap_list) + 8ll * cap_rows * d +
         8ll * cap_rows;
}
__global__ void plan_kernel(const ure_mf_shard_t* shards, int K, int batch, int avail_smem, OwnerWs* ws) {
  __shared__ PlanScratch ps;
  __shared__ Plan pl;
  make_plan(shards, K, blockIdx.x, gridDim.x, pl, ps);
  if (threadIdx.x == 0) {
    if (blockIdx.x == 0) ws->avail_smem = avail_smem;
    atomicMax(&ws->max_rows, (pl.ru1 - pl.ru0) + (pl.ri1 - pl.ri0));
    atomicMax(&ws->max_slots, pl.mU + pl.mI);
    atomicMax(&ws->max_spe, (shards[pl.shard].n + batch - 1) / batch);
    if (blockIdx.x == 0) {
      long long tot = 0;
      for (int s = 0; s < K; ++s) tot += 2ll * shards[s].n;
      ws->tot_slots = tot;
    }
  }
}

// ---------------------------------------------------------------- set-up: the records sorted by user / by item
// Row offsets: histogram + scan.  Records: a STABLE least-significant-digit radix sort on the row number (8-bit
// digits), so the records of a row stay in record order and the whole training is reproducible bit for bit
// (the gradient of a row is summed in slot order).  Pass p of side (user | item) reads the shard's records
// (p = 0) or the previous pass's output and writes the other of {tmp, final}; the last pass lands in final.
// smem_rows > 0: the shard's rows (user + item) fit a shared-memory histogram of that many counters -- the global
// atomics (875 k x 2 on a few thousand hot addresses at ml1m size) shrink to one per row and CTA
// Rating files are written user by user (ML-1M / ML-20M, and what readRating hands over), so a shard's records usually
// arrive ALREADY in user-row order and the stable sort by user is the identity.  The counting pass checks that while
// it reads the records (every record against its predecessor) and writes the user-sorted copy speculatively
// (inter_u[j] = record j, pad = j): when no inversion shows up, the radix passes of the user side return at once
// (ws->unsorted[shard] == 0); otherwise they overwrite the copy.  Same bytes either way.
__device__ __forceinline__ void note_order(const ure_mf_shard_t& sh, long long j, const int4& r, unsigned* unsorted) {
  if (!unsorted) return;
  if (j > 0 && __ldg(&sh.inter[j - 1].user) > r.x) *unsorted = 1u;      // benign race: every writer stores 1
  reinterpret_cast<int4*>(sh.inter_u)[j] = make_int4(r.x, r.y, r.z, (int)j);
}

// virtual block (bx of gx, shard by); s_cnt: smem_rows ints (or unused)
__device__ __forceinline__ void csr_count_body(const ure_mf_shard_t* shards, int smem_rows, unsigned* unsorted_flags,
                                               int* s_cnt, int bx, int by, int gx) {
  const ure_mf_shard_t& sh = shards[by];
  const long long stride = (long long)gx * blockDim.x;
  const int nu = sh.n_user, rows = sh.n_user + sh.n_item;
  unsigned* const unsorted = unsorted_flags ? unsorted_flags + by : nullptr;
  if (smem_rows > 0 && rows <= smem_rows) {
    for (int x = threadIdx.x; x < rows; x += blockDim.x) s_cnt[x] = 0;
    __syncthreads();
    for (long long j = (long long)bx * blockDim.x + threadIdx.x; j < sh.n; j += stride) {
      const int4 r = ld_stream_i4(sh.inter + j);
      atomicAdd(&s_cnt[r.x], 1);
      atomicAdd(&s_cnt[nu + r.y], 1);
      note_order(sh, j, r, unsorted);
    }
    __syncthreads();
    for (int x = threadIdx.x; x < rows; x += blockDim.x) {
      const int c = s_cnt[x];
      if (c) atomicAdd(x < nu ? sh.off_u + x + 1 : sh.off_i + (x - nu) + 1, c);
    }
    return;
  }
  for (long long j = (long long)bx * blockDim.x + threadIdx.x; j < sh.n; j += stride) {
    const int4 r = ld_stream_i4(sh.inter + j);
    atomicAdd(sh.off_u + r.x + 1, 1);
    atomicAdd(sh.off_i + r.y + 1, 1);
    note_order(sh, j, r, unsorted);
  }
}

__global__ void csr_count_kernel(const ure_mf_shard_t* shards, int smem_rows, unsigned* unsorted_flags) {
  extern __shared__ int s_cnt[];
  csr_count_body(shards, smem_rows, unsorted_flags, s_cnt, blockIdx.x, blockIdx.y, gridDim.x);
}

// in-place inclusive scan of off[0 .. rows+2): one CTA per (shard, side); off[r] becomes the first slot of row r
// s_scr: 33 ints of shared memory
__device__ __forceinline__ void csr_scan_body(const ure_mf_shard_t* shards, int* s_scr, int vb) {
  const ure_mf_shard_t& sh = shards[vb >> 1];
  int32_t* off = (vb & 1) ? sh.off_i : sh.off_u;
  const int len = ((vb & 1) ? sh.n_item : sh.n_user) + 2;
  int* const s_warp = s_scr;
  int& s_carry = s_scr[32];
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int base = 0; base < len; base += blockDim.x) {
    const int x = base + threadIdx.x;
    int v = x < len ? off[x] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int a = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += a;
    }
    if (lane == 31) s_warp[warp] = v;
    __syncthreads();
    if (warp == 0) {
      int w = lane < (int)(blockDim.x >> 5) ? s_warp[lane] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int a = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += a;
      }
      s_warp[lane] = w;
    }
    __syncthreads();
    const int carry = s_carry + (warp > 0 ? s_warp[warp - 1] : 0);
    if (x < len) off[x] = v + carry;
    __syncthreads();
    if (threadIdx.x == 0) s_carry += s_warp[31];
    __syncthreads();
  }
}

__global__ void csr_scan_kernel(const ure_mf_shard_t* shards) {
  __shared__ int s_scr[33];
  csr_scan_body(shards, s_scr, blockIdx.x);
}

constexpr int kRadixBlocks = 96;          // CTAs per (shard, side): each owns a contiguous tile of the records
constexpr int kRadixThreads = 512;
constexpr int kRadixWarps = kRadixThreads / 32;

struct RadixView {                        // what pass `pass` of virtual block (bx of gx, by = 2*shard + side) works on
  const int4* src;
  int4* dst;
  long long n, t0, t1;                    // the CTA's tile [t0, t1)
  bool item, first;
  __device__ RadixView(const ure_mf_shard_t* shards, int pass, int npass, int bx, int by, int gx) {
    const ure_mf_shard_t& sh = shards[by >> 1];
    item = by & 1;
    first = pass == 0;
    int4* fin = reinterpret_cast<int4*>(item ? sh.inter_i : sh.inter_u);
    int4* tmp = reinterpret_cast<int4*>(item ? sh.tmp_i : sh.tmp_u);
    dst = ((npass - 1 - pass) & 1) ? tmp : fin;
    src = first ? reinterpret_cast<const int4*>(sh.inter) : (((npass - pass) & 1) ? tmp : fin);
    n = sh.n;
    const long long tile = (n + gx - 1) / gx;
    t0 = min(n, tile * bx);
    t1 = min(n, t0 + tile);
  }
  __device__ __forceinline__ int digit(const int4& r, int pass) const { return ((item ? r.y : r.x) >> (8 * pass)) & 255; }
};

// hist [2 * shards][gx][256]: records of the CTA's tile per digit value.  s_h: 256 ints.  Any block size (multiple of 32).
__device__ __forceinline__ void radix_hist_body(const ure_mf_shard_t* shards, int pass, int npass, int* __restrict__ hist,
                                                const unsigned* unsorted, int* s_h, int bx, int by, int gx) {
  if (unsorted && !(by & 1) && unsorted[by >> 1] == 0) return;      // user side already in order
  const RadixView v(shards, pass, npass, bx, by, gx);
  for (int x = threadIdx.x; x < 256; x += blockDim.x) s_h[x] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  for (long long j0 = v.t0 + (threadIdx.x & ~31); j0 < v.t1; j0 += blockDim.x) {      // warp-uniform trip count
    const long long j = j0 + lane;
    const bool in = j < v.t1;
    const int dg = in ? v.digit(__ldg(v.src + j), pass) : 0;
    const unsigned act = __ballot_sync(0xffffffffu, in);
    if (in) {
      const unsigned same = __match_any_sync(act, dg);
      if (lane == __ffs(same) - 1) atomicAdd(&s_h[dg], __popc(same));
    }
  }
  __syncthreads();
  for (int x = threadIdx.x; x < 256; x += blockDim.x) hist[((long long)by * gx + bx) * 256 + x] = s_h[x];
}

__global__ void __launch_bounds__(kRadixThreads)
radix_hist_kernel(const ure_mf_shard_t* shards, int pass, int npass, int* __restrict__ hist, const unsigned* unsorted) {
  __shared__ int s_h[256];
  radix_hist_body(shards, pass, npass, hist, unsorted, s_h, blockIdx.x, blockIdx.y, gridDim.x);
}

// per row y = 2 * shard + side: exclusive scan of hist in (digit, CTA) order, in place; threads 0..255 of one CTA per y.
// s_tot: 256 ints.
__device__ __forceinline__ void radix_scan_body(int* __restrict__ hist, int n_blocks, const unsigned* unsorted, int* s_tot, int y) {
  if (unsorted && !(y & 1) && unsorted[y >> 1] == 0) return;
  const bool on = threadIdx.x < 256;
  int* h = hist + (long long)y * n_blocks * 256 + (threadIdx.x & 255);      // thread = digit: coalesced per CTA row
  if (on) {
    int tot = 0;
    for (int b = 0; b < n_blocks; ++b) tot += h[b * 256];
    s_tot[threadIdx.x] = tot;
  }
  __syncthreads();
  if (threadIdx.x < 32) {                 // exclusive scan of the 256 digit totals by one warp, 8 per lane
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
  if (on) {
    int run = s_tot[threadIdx.x];
    for (int b = 0; b < n_blocks; ++b) {
      const int t = h[b * 256];
      h[b * 256] = run;
      run += t;
    }
  }
}

__global__ void __launch_bounds__(256)
radix_scan_kernel(int* __restrict__ hist, int n_blocks, const unsigned* unsorted) {
  __shared__ int s_tot[256];
  radix_scan_body(hist, n_blocks, unsorted, s_tot, blockIdx.x);
}

// stable scatter of the CTA's tile: every warp owns a contiguous range; per-warp digit counts -> per-warp cursors
// (from the CTA's global offsets); inside a warp __match_any ranks the lanes of one digit in lane (= record) order.
// s_whp: [kRadixWarps][256] ints; block size kRadixThreads.
__device__ __forceinline__ void radix_scatter_body(const ure_mf_shard_t* shards, int pass, int npass, const int* __restrict__ hist,
                                                   const unsigned* unsorted, int* s_whp, int bx, int by, int gx) {
  if (unsorted && !(by & 1) && unsorted[by >> 1] == 0) return;
  int (*s_wh)[256] = reinterpret_cast<int (*)[256]>(s_whp);
  const RadixView v(shards, pass, npass, bx, by, gx);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned lt = (1u << lane) - 1u;
  for (int x = threadIdx.x; x < kRadixWarps * 256; x += blockDim.x) s_whp[x] = 0;
  __syncthreads();
  const long long per = ((v.t1 - v.t0) + kRadixWarps - 1) / kRadixWarps;
  const long long w0 = min(v.t1, v.t0 + per * warp), w1 = min(v.t1, w0 + per);
  for (long long j0 = w0; j0 < w1; j0 += 32) {
    const long long j = j0 + lane;
    const bool in = j < w1;
    const int dg = in ? v.digit(__ldg(v.src + j), pass) : 0;
    const unsigned act = __ballot_sync(0xffffffffu, in);
    if (in) {
      const unsigned same = __match_any_sync(act, dg);
      if (lane == __ffs(same) - 1) s_wh[warp][dg] += __popc(same);        // the warp's own counters
    }
    __syncwarp();
  }
  __syncthreads();
  if (threadIdx.x < 256) {
    int run = hist[((long long)by * gx + bx) * 256 + threadIdx.x];
    for (int w = 0; w < kRadixWarps; ++w) {
      const int t = s_wh[w][threadIdx.x];
      s_wh[w][threadIdx.x] = run;
      run += t;
    }
  }
  __syncthreads();
  for (long long j0 = w0; j0 < w1; j0 += 32) {
    const long long j = j0 + lane;
    const bool in = j < w1;
    int4 r = make_int4(0, 0, 0, 0);
    if (in) {
      r = __ldg(v.src + j);
      if (v.first) r.w = (int)j;          // the record's index in the shard's own order
    }
    const int dg = v.digit(r, pass);
    const unsigned act = __ballot_sync(0xffffffffu, in);
    if (in) {
      const unsigned same = __match_any_sync(act, dg);
      v.dst[s_wh[warp][dg] + __popc(same & lt)] = r;
      __syncwarp(act);
      if (lane == __ffs(same) - 1) s_wh[warp][dg] += __popc(same);
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(kRadixThreads)
radix_scatter_kernel(const ure_mf_shard_t* shards, int pass, int npass, const int* __restrict__ hist, const unsigned* unsorted) {
  __shared__ int s_wh[kRadixWarps * 256];
  radix_scatter_body(shards, pass, npass, hist, unsorted, s_wh, blockIdx.x, blockIdx.y, gridDim.x);
}

// The whole set-up in ONE cooperative launch (batches whose set-up is launch-bound: eight launches of a few
// microseconds each): the bodies above run as virtual blocks of a co-resident grid, with a grid barrier where a launch
// boundary was.  Dynamic shared memory: max(smem_rows, kRadixWarps * 256) ints.
//   count + histogram of pass 0 | row-offset scan + digit scan | scatter | histogram | digit scan | scatter ...
// The bodies read their source records with __ldg although a later pass reads what an earlier pass of THIS launch
// wrote: up to three passes (rows < 2^24) no buffer is read through the non-coherent path, rewritten and read again
// inside the launch (pass p reads only what pass p - 1 wrote into a buffer nobody has read yet), and every grid barrier
// ends in an acquire that drops the SM's L1 lines anyway.
__global__ void __launch_bounds__(kRadixThreads)
owner_setup_kernel(const ure_mf_shard_t* shards, int n_shards, int smem_rows, int cb, int npass, int* __restrict__ hist,
                   unsigned* unsorted) {
  extern __shared__ int s_dyn[];
  cg::grid_group grid = cg::this_grid();
  const int G = gridDim.x, me = blockIdx.x;
  const int n_count = cb * n_shards, n_radix = kRadixBlocks * 2 * n_shards, n_scan = 2 * n_shards;
  // the histogram blocks of pass 0 first (they do not depend on the counting pass): the user side is counted although
  // the records may turn out to be in user order already -- the flags are final only at the first barrier
  for (int vb = me; vb < n_radix + n_count; vb += G) {
    if (vb < n_count) csr_count_body(shards, smem_rows, unsorted, s_dyn, vb % cb, vb / cb, cb);      // the longer blocks first
    else radix_hist_body(shards, 0, npass, hist, nullptr, s_dyn, (vb - n_count) % kRadixBlocks, (vb - n_count) / kRadixBlocks, kRadixBlocks);
    __syncthreads();
  }
  for (int pass = 0; pass < npass; ++pass) {
    if (pass > 0) {
      grid.sync();
      for (int vb = me; vb < n_radix; vb += G) {
        radix_hist_body(shards, pass, npass, hist, unsorted, s_dyn, vb % kRadixBlocks, vb / kRadixBlocks, kRadixBlocks);
        __syncthreads();
      }
    }
    grid.sync();
    for (int vb = me; vb < n_scan * (pass == 0 ? 2 : 1); vb += G) {
      if (vb < n_scan) radix_scan_body(hist, kRadixBlocks, unsorted, s_dyn, vb);
      else csr_scan_body(shards, s_dyn, vb - n_scan);
      __syncthreads();
    }
    grid.sync();
    for (int vb = me; vb < n_radix; vb += G) {
      radix_scatter_body(shards, pass, npass, hist, unsorted, s_dyn, vb % kRadixBlocks, vb / kRadixBlocks, kRadixBlocks);
      __syncthreads();
    }
  }
}

__global__ void perm_inverse_kernel(const ure_mf_shard_t* shards, int epochs) {
  const ure_mf_shard_t& sh = shards[blockIdx.y];
  if (!sh.perm || !sh.perm_inv) return;
  const long long total = (long long)epochs * sh.n;
  for (long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += (long long)gridDim.x * blockDim.x) {
    const long long e = x / sh.n;
    sh.perm_inv[e * sh.n + sh.perm[x]] = (int32_t)(x - e * sh.n);
  }
}

// ---------------------------------------------------------------- the schedule pre-pass
// Block (cta, y): for the training CTA `cta` and the rows r = y, y + gridDim.y, ... of the window that starts at
// global step step0 (row r = epoch step0 / spe + r of the CTA's shard): the CTA's slots, stably sorted by the step
// whose batch they are in.
//   sched [rows][stride] u16 : row r, positions slot_base .. slot_base + m
//   off   [rows][grid][spe_cap + 1] int : start of every step's run inside the CTA's m entries (off[spe] = m)
constexpr int kSchedThreads = 512;
constexpr int kSchedWarps = kSchedThreads / 32;

__host__ __device__ inline long long schedule_smem_bytes(int cap_slots, int spe_cap, bool cache_j, int tab_cap = 0) {
  // record index of every slot [cap] int (optional) | step of every slot [cap] u16 | rank of every slot [cap] u16
  // (short epochs only) | histogram [spe_cap + 1] int | per-warp bin counters [warps][64] int | 4 round-function
  // tables [tab_cap] u16 (optional)
  return (cache_j ? 4ll : 0ll) * cap_slots + 2ll * cap_slots + (spe_cap <= 64 ? 2ll * cap_slots : 0ll) +
         4ll * (spe_cap + 1) + 4ll * kSchedWarps * 64 + 16 + 8ll * tab_cap;
}
constexpr int kTabMaxHalf = 8192;         // round tables: a, b <= this (n <= 6.7e7)

__global__ void __launch_bounds__(kSchedThreads, 2)
owner_schedule_kernel(const ure_mf_shard_t* __restrict__ shards, int K, ure_mf_hparams_t hp, int epochs,
                      long long step0, int tab_cap) {
  constexpr int NW = kSchedWarps;
  constexpr unsigned FULL = 0xffffffffu;
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ PlanScratch s_ps;
  __shared__ Plan s_pl;
  __shared__ int s_warp_tot[NW];
  __shared__ int s_carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  make_plan(shards, K, blockIdx.x, gridDim.x, s_pl, s_ps);
  const ure_mf_shard_t& sh = shards[s_pl.shard];
  const int mU = s_pl.mU, m = mU + s_pl.mI;
  const int B = hp.batch, n = sh.n;
  const int spe = (n + B - 1) / B;
  if (plan_not_covered(hp, s_pl, spe)) return;
  if (spe == 0) return;
  const int cap = hp.owner_cap_slots, spe_cap = hp.owner_spe_cap;
  const bool cache_j = (hp.owner_flags & 2) == 0, short_ok = spe_cap <= 64;
  int* const s_j = reinterpret_cast<int*>(dyn);                            // [cap] record index of the slot
  unsigned short* const s_stepof = reinterpret_cast<unsigned short*>(s_j + (cache_j ? cap : 0));
  unsigned short* const s_rank = s_stepof + cap;                           // [cap] rank inside (warp, step)
  int* const s_hist = reinterpret_cast<int*>(s_rank + (short_ok ? cap : 0));   // [spe_cap + 1]
  int* const s_wh = s_hist + spe_cap + 1;                                  // [NW][64]
  // tab_cap > 0: a Feistel round adds f_r(other half) to one half, and the halves live in [0, a) / [0, b) with
  // a, b ~ sqrt(n): the four round functions of an epoch are TABLES (2 (a + b) u16, built by the CTA per epoch), so
  // a round of the inverse network is one shared-memory load, a compare and an add instead of two multiplies, a
  // shift, an xor and a mulhi
  unsigned short* const s_tab = reinterpret_cast<unsigned short*>(s_wh + NW * 64 + 4);     // 4 x [tab_cap]
  const int4* const recU = reinterpret_cast<const int4*>(sh.inter_u + s_pl.su0);
  const int4* const recI = reinterpret_cast<const int4*>(sh.inter_i + s_pl.si0) - mU;
  if (cache_j)
    for (int sl = tid; sl < m; sl += kSchedThreads) s_j[sl] = __ldg(&((sl >= mU ? recI : recU) + sl)->w);
  FeistelDomain dom;
  dom.init((uint32_t)n);
  const uint32_t magic = (uint32_t)(0x100000000ull / (uint32_t)B);         // floor(2^32/B): quotient low by <= 1
  const int per = (m + NW - 1) / NW;                                       // every warp owns a contiguous range
  const int w0 = min(warp * per, m), w1 = min(w0 + per, m);
  const unsigned lt = (1u << lane) - 1u;

  for (int r = blockIdx.y; r < hp.owner_sched_rows; r += gridDim.y) {
    const int epoch = (int)(step0 / spe) + r;
    if (epoch >= epochs) break;
    unsigned short* const out = hp.owner_sched + (long long)r * hp.owner_sched_stride + s_pl.slot_base;
    int* const off = hp.owner_sched_off + ((long long)r * gridDim.x + blockIdx.x) * (spe_cap + 1);
    FeistelKeys ks;
    ks.init(perm_key(sh.perm_seed, (uint32_t)sh.shard_id, (uint32_t)epoch));
    const int32_t* pinv = sh.perm_inv ? sh.perm_inv + (long long)epoch * n : nullptr;
    constexpr int NI = 4;
    const bool tabbed = tab_cap > 0 && !pinv && n > 1;
    if (tabbed) {
      __syncthreads();                     // the previous row is done with the tables
      for (int x = tid; x < (int)dom.b; x += kSchedThreads) {
        s_tab[x] = (unsigned short)mulhi32(round_hash((uint32_t)x ^ ks.rk[0]), dom.a);
        s_tab[2 * tab_cap + x] = (unsigned short)mulhi32(round_hash((uint32_t)x ^ ks.rk[2]), dom.a);
      }
      for (int x = tid; x < (int)dom.a; x += kSchedThreads) {
        s_tab[tab_cap + x] = (unsigned short)mulhi32(round_hash((uint32_t)x ^ ks.rk[1]), dom.b);
        s_tab[3 * tab_cap + x] = (unsigned short)mulhi32(round_hash((uint32_t)x ^ ks.rk[3]), dom.b);
      }
      // (the __syncthreads that every path below starts with publishes the tables)
    }
    // step of NI x 32 consecutive slots of this warp's range (lane = slot inside a 32-block)
    auto steps_of = [&](int base, uint32_t (&q)[NI], bool (&live)[NI]) {
      uint32_t x[NI];
#pragma unroll
      for (int u = 0; u < NI; ++u) {
        const int sl = base + 32 * u + lane;
        live[u] = sl < w1;
        x[u] = !live[u] ? 0u : cache_j ? (uint32_t)s_j[sl] : (uint32_t)__ldg(&((sl >= mU ? recI : recU) + sl)->w);
      }
      if (pinv) {
#pragma unroll
        for (int u = 0; u < NI; ++u)
          if (live[u]) x[u] = (uint32_t)__ldg(pinv + x[u]);
      } else if (tabbed) {
        const unsigned short* const T0 = s_tab, *const T1 = s_tab + tab_cap, *const T2 = s_tab + 2 * tab_cap,
                                    *const T3 = s_tab + 3 * tab_cap;
        bool pend[NI];
#pragma unroll
        for (int u = 0; u < NI; ++u) pend[u] = live[u];
        bool any = true;
        while (any) {                      // cycle walking: almost never a second trip
          uint32_t L[NI], R[NI];
#pragma unroll
          for (int u = 0; u < NI; ++u) dom.split(x[u], L[u], R[u]);
#pragma unroll
          for (int u = 0; u < NI; ++u) { const uint32_t f = T3[L[u]]; R[u] = R[u] >= f ? R[u] - f : R[u] + dom.b - f; }
#pragma unroll
          for (int u = 0; u < NI; ++u) { const uint32_t f = T2[R[u]]; L[u] = L[u] >= f ? L[u] - f : L[u] + dom.a - f; }
#pragma unroll
          for (int u = 0; u < NI; ++u) { const uint32_t f = T1[L[u]]; R[u] = R[u] >= f ? R[u] - f : R[u] + dom.b - f; }
#pragma unroll
          for (int u = 0; u < NI; ++u) { const uint32_t f = T0[R[u]]; L[u] = L[u] >= f ? L[u] - f : L[u] + dom.a - f; }
          any = false;
#pragma unroll
          for (int u = 0; u < NI; ++u) {
            if (pend[u]) {
              x[u] = L[u] * dom.b + R[u];
              pend[u] = x[u] >= dom.n;
              any |= pend[u];
            }
          }
        }
      } else {
        feistel_inverse_n<NI>(dom, ks, x, live);
      }
#pragma unroll
      for (int u = 0; u < NI; ++u) {
        q[u] = B == 1 ? x[u] : mulhi32(x[u], magic);
        if ((q[u] + 1) * (uint32_t)B <= x[u]) ++q[u];
      }
    };
    if (spe <= 64 && short_ok) {
      // ---- short epochs (the common case): ONE pass computes the steps and the per-warp bin counts, two warps
      // turn them into cursors, one pass scatters
      for (int x = tid; x < NW * 64; x += kSchedThreads) s_wh[x] = 0;
      __syncthreads();                     // also: s_j complete, the previous row's scatter done
      for (int base = w0; base < w1; base += 32 * NI) {
        uint32_t q[NI];
        bool live[NI];
        steps_of(base, q, live);
#pragma unroll
        for (int u = 0; u < NI; ++u) {     // rank of the slot among the warp's slots of the same step, in slot order
          const unsigned act = __ballot_sync(FULL, live[u]);
          unsigned same = 0;
          int old = 0;
          if (live[u]) {
            same = __match_any_sync(act, q[u]);
            old = s_wh[warp * 64 + q[u]];                  // the warp's own counters
            s_stepof[base + 32 * u + lane] = (unsigned short)q[u];
            s_rank[base + 32 * u + lane] = (unsigned short)(old + __popc(same & lt));
          }
          __syncwarp();
          if (live[u] && lane == __ffs(same) - 1) s_wh[warp * 64 + q[u]] = old + __popc(same);
          __syncwarp();
        }
      }
      __syncthreads();
      if (tid < 64) {                      // bin totals -> bin starts (two warps) -> per-warp bases
        int tot = 0;
        for (int w = 0; w < NW; ++w) tot += s_wh[w * 64 + tid];
        int inc = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int a = __shfl_up_sync(FULL, inc, o);
          if (lane >= o) inc += a;
        }
        if (tid == 31) s_carry = inc;
        asm volatile("bar.sync 1, 64;" ::: "memory");
        int run = inc - tot + (tid >= 32 ? s_carry : 0);
        if (tid <= spe) off[tid] = tid < spe ? run : m;
        if (tid == 63 && spe == 64) off[64] = m;
        for (int w = 0; w < NW; ++w) {
          const int t = s_wh[w * 64 + tid];
          s_wh[w * 64 + tid] = run;
          run += t;
        }
      }
      __syncthreads();
      for (int sl = w0 + lane; sl < w1; sl += 32)            // position = base of (warp, step) + rank: no order needed
        out[s_wh[warp * 64 + s_stepof[sl]] + s_rank[sl]] = (unsigned short)sl;
      __syncthreads();
      continue;
    }
    // ---- long epochs: histogram over all steps, then the scatter in groups of 64 steps
    for (int b = tid; b <= spe; b += kSchedThreads) s_hist[b] = 0;
    __syncthreads();                       // also: s_j complete, the previous row's scatter done
    for (int base = w0; base < w1; base += 32 * NI) {
      uint32_t q[NI];
      bool live[NI];
      steps_of(base, q, live);
#pragma unroll
      for (int u = 0; u < NI; ++u) {
        const unsigned act = __ballot_sync(FULL, live[u]);
        if (live[u]) {
          s_stepof[base + 32 * u + lane] = (unsigned short)q[u];
          const unsigned same = __match_any_sync(act, q[u]);
          if (lane == __ffs(same) - 1) atomicAdd(&s_hist[q[u]], __popc(same));
        }
        __syncwarp();
      }
    }
    __syncthreads();
    // ---- exclusive scan of the histogram (spe + 1 entries, the last becomes m)
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base <= spe; base += kSchedThreads) {
      const int x = base + tid;
      const int v = x <= spe ? s_hist[x] : 0;
      int inc = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int a = __shfl_up_sync(FULL, inc, o);
        if (lane >= o) inc += a;
      }
      if (lane == 31) s_warp_tot[warp] = inc;
      __syncthreads();
      if (warp == 0) {
        int w = lane < NW ? s_warp_tot[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int a = __shfl_up_sync(FULL, w, o);
          if (lane >= o) w += a;
        }
        if (lane < NW) s_warp_tot[lane] = w;
      }
      __syncthreads();
      const int excl = s_carry + (warp > 0 ? s_warp_tot[warp - 1] : 0) + inc - v;
      if (x <= spe) { s_hist[x] = excl; off[x] = excl; }
      __syncthreads();
      if (tid == 0) s_carry += s_warp_tot[NW - 1];
      __syncthreads();
    }
    // ---- stable scatter, 64 steps at a time: per-warp bin counts -> per-warp bin cursors; inside a warp
    // __match_any ranks the lanes of one bin in lane (= slot) order
    for (int g0 = 0; g0 < spe; g0 += 64) {
      for (int x = tid; x < NW * 64; x += kSchedThreads) s_wh[x] = 0;
      __syncthreads();
      for (int s0 = w0; s0 < w1; s0 += 32) {
        const int sl = s0 + lane;
        const int b = sl < w1 ? (int)s_stepof[sl] - g0 : -1;
        const bool in = b >= 0 && b < 64;
        const unsigned act = __ballot_sync(FULL, in);
        if (in) {
          const unsigned same = __match_any_sync(act, b);
          if (lane == __ffs(same) - 1) s_wh[warp * 64 + b] += __popc(same);     // the warp's own counters
        }
        __syncwarp();
      }
      __syncthreads();
      if (tid < 64 && g0 + tid < spe) {
        int run = s_hist[g0 + tid];
        for (int w = 0; w < NW; ++w) {
          const int t = s_wh[w * 64 + tid];
          s_wh[w * 64 + tid] = run;
          run += t;
        }
      }
      __syncthreads();
      for (int s0 = w0; s0 < w1; s0 += 32) {
        const int sl = s0 + lane;
        const int b = sl < w1 ? (int)s_stepof[sl] - g0 : -1;
        const bool in = b >= 0 && b < 64;
        const unsigned act = __ballot_sync(FULL, in);
        if (in) {
          const unsigned same = __match_any_sync(act, b);
          out[s_wh[warp * 64 + b] + __popc(same & lt)] = (unsigned short)sl;
          __syncwarp(act);
          if (lane == __ffs(same) - 1) s_wh[warp * 64 + b] += __popc(same);
        }
        __syncwarp();
      }
      __syncthreads();
    }
  }
}

// ---------------------------------------------------------------- the schedule pre-pass, short epochs (the usual case)
// Same output as owner_schedule_kernel for epochs of at most 64 steps, at half its instruction count and shared memory
// (two CTAs per SM instead of one; ncu of the general kernel: 136 warp-instructions per 32 slots and epoch, one CTA
// per SM because of 117 KB of shared memory, issue slots 45 % busy):
//   * the (L, R) halves of a slot's record index -- what every epoch's inverse network starts from -- are split once
//     per launch and kept as one packed word per slot, in doubled units so that a half IS the byte offset into a
//     16-bit round table;
//   * the four rounds of the inverse network read a per-epoch table (one LDS of random lanes: ~3.5 bank wavefronts);
//   * cycle walking (x >= n, one slot in ~400) is a rare divergent loop instead of a second trip of the whole group;
//   * step and rank of a slot share one 16-bit word; the per-(step, warp) counts are scanned by the whole CTA.
// Lists are identical to the general kernel's (same stable order), so either serves the training kernel.
__host__ __device__ inline long long schedule_tab_smem_bytes(int cap_slots, int tab_cap) {
  // packed halves / record index [cap] u32 | step + rank [cap] u16 | counters [warps][64] int | scan scratch |
  // round tables 2 sets x 4 x [tab_cap] u16
  return 4ll * cap_slots + 2ll * cap_slots + 4ll * kSchedWarps * 64 + 4ll * (kSchedWarps + 4) + 2ll * 2 * 4 * tab_cap + 64;
}

__global__ void __maxnreg__(64)
owner_schedule_tab_kernel(const ure_mf_shard_t* __restrict__ shards, int K, ure_mf_hparams_t hp, int epochs,
                          long long step0, int tab_cap, int sb) {
  constexpr int NW = kSchedWarps;
  constexpr unsigned FULL = 0xffffffffu;
  constexpr int NI = 4;
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ PlanScratch s_ps;
  __shared__ Plan s_pl;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  make_plan(shards, K, blockIdx.x, gridDim.x, s_pl, s_ps);
  const ure_mf_shard_t& sh = shards[s_pl.shard];
  const int mU = s_pl.mU, m = mU + s_pl.mI;
  const int B = hp.batch, n = sh.n;
  const int spe = (n + B - 1) / B;
  if (plan_not_covered(hp, s_pl, spe)) return;
  if (spe == 0) return;
  const int cap = hp.owner_cap_slots, spe_cap = hp.owner_spe_cap;
  uint32_t* const s_lr = reinterpret_cast<uint32_t*>(dyn);                       // [cap] packed halves / record index
  unsigned short* const s_sr = reinterpret_cast<unsigned short*>(s_lr + cap);    // [cap] step | rank << sb
  int* const s_wh = reinterpret_cast<int*>(s_sr + cap);                          // [NW][64]
  int* const s_wtot = s_wh + NW * 64;                                            // [NW + 4]
  unsigned char* const s_tab = reinterpret_cast<unsigned char*>(s_wtot + NW + 4);   // 2 sets x 4 x [tab_cap] u16
  const uint32_t tab_bytes = 2u * (uint32_t)tab_cap;
  const int4* const recU = reinterpret_cast<const int4*>(sh.inter_u + s_pl.su0);
  const int4* const recI = reinterpret_cast<const int4*>(sh.inter_i + s_pl.si0) - mU;
  FeistelDomain dom;
  dom.init((uint32_t)n);
  const bool explicit_order = sh.perm_inv != nullptr;
  const bool trivial = n <= 1;
  for (int sl = tid; sl < m; sl += kSchedThreads) {
    const uint32_t j = (uint32_t)__ldg(&((sl >= mU ? recI : recU) + sl)->w);
    uint32_t L, R;
    dom.split(j, L, R);
    s_lr[sl] = explicit_order || trivial ? j : (L << 17) | (R << 1);
  }
  const uint32_t B2 = 2u * (uint32_t)B;
  const uint32_t magic2 = (uint32_t)(0x100000000ull / B2);                       // floor(2^32 / 2B): quotient low by <= 1
  const uint32_t a2 = 2u * dom.a, b2 = 2u * dom.b, n2 = 2u * dom.n;
  const int per = ((m + NW - 1) / NW + 31) & ~31;                                // whole 32-slot blocks per warp
  const int w0 = min(warp * per, m), w1 = min(w0 + per, m);
  const unsigned lt = (1u << lane) - 1u;
  const uint32_t qmask = (1u << sb) - 1u;

  // round tables of one epoch (rounds 3, 2, 1, 0), doubled values, built by threads t0, t0 + nthr, ... of the CTA
  auto build_tables = [&](int epoch, unsigned char* tab, int t0, int nthr) {
    if (explicit_order || trivial || t0 < 0) return;
    FeistelKeys kt;
    kt.init(perm_key(sh.perm_seed, (uint32_t)sh.shard_id, (uint32_t)epoch));
    for (int x = t0; x < (int)dom.a; x += nthr) {
      *reinterpret_cast<unsigned short*>(tab + 2 * x) = (unsigned short)(2u * mulhi32(round_hash((uint32_t)x ^ kt.rk[3]), dom.b));
      *reinterpret_cast<unsigned short*>(tab + 2 * tab_bytes + 2 * x) = (unsigned short)(2u * mulhi32(round_hash((uint32_t)x ^ kt.rk[1]), dom.b));
    }
    for (int x = t0; x < (int)dom.b; x += nthr) {
      *reinterpret_cast<unsigned short*>(tab + tab_bytes + 2 * x) = (unsigned short)(2u * mulhi32(round_hash((uint32_t)x ^ kt.rk[2]), dom.a));
      *reinterpret_cast<unsigned short*>(tab + 3 * tab_bytes + 2 * x) = (unsigned short)(2u * mulhi32(round_hash((uint32_t)x ^ kt.rk[0]), dom.a));
    }
  };
  const int e_first = (int)(step0 / spe);
  if (blockIdx.y < hp.owner_sched_rows && e_first + (int)blockIdx.y < epochs) build_tables(e_first + blockIdx.y, s_tab, tid, kSchedThreads);
  for (int x = tid; x < NW * 64; x += kSchedThreads) s_wh[x] = 0;
  __syncthreads();

  int it = 0;
  for (int r = blockIdx.y; r < hp.owner_sched_rows; r += gridDim.y, ++it) {
    const int epoch = e_first + r;
    if (epoch >= epochs) break;
    unsigned short* const out = hp.owner_sched + (long long)r * hp.owner_sched_stride + s_pl.slot_base;
    int* const off = hp.owner_sched_off + ((long long)r * gridDim.x + blockIdx.x) * (spe_cap + 1);
    const int32_t* const pinv = explicit_order ? sh.perm_inv + (long long)epoch * n : nullptr;
    const unsigned char* const tabs = s_tab + (it & 1) * 4 * tab_bytes;         // tables alternate between two sets
    // one round of the inverse network in doubled units: h -= 2 f(o) (mod m2)
    auto round_tab = [&](uint32_t& h, uint32_t o2, uint32_t t, uint32_t m2) {
      const uint32_t f = *reinterpret_cast<const unsigned short*>(tabs + t * tab_bytes + o2);
      const uint32_t d = h - f;
      h = min(d, d + m2);                  // unsigned: the wrapped difference is the larger one
    };
    auto inverse2 = [&](uint32_t Ls, uint32_t Rs) {       // -> 2 x position
      round_tab(Rs, Ls, 0, b2); round_tab(Ls, Rs, 1, a2);
      round_tab(Rs, Ls, 2, b2); round_tab(Ls, Rs, 3, a2);
      return (Ls >> 1) * b2 + Rs;
    };
    // ---- pass 1: step of every slot; rank among the warp's slots of the same step, in slot order.  No CTA barrier
    // since the previous row's pass 2: a warp touches its own range of s_sr and its own counters only
    for (int base = w0; base < w1; base += 32 * NI) {
      uint32_t x2[NI];
      bool live[NI];
#pragma unroll
      for (int u = 0; u < NI; ++u) {
        const int sl = base + 32 * u + lane;
        live[u] = sl < w1;
        x2[u] = live[u] ? s_lr[sl] : 0u;
      }
      if (explicit_order) {
#pragma unroll
        for (int u = 0; u < NI; ++u) x2[u] = live[u] ? 2u * (uint32_t)__ldg(pinv + x2[u]) : 0u;
      } else if (trivial) {
#pragma unroll
        for (int u = 0; u < NI; ++u) x2[u] = 0u;
      } else {
#pragma unroll
        for (int u = 0; u < NI; ++u) x2[u] = inverse2(x2[u] >> 16, x2[u] & 0xffffu);
#pragma unroll
        for (int u = 0; u < NI; ++u)
          while (x2[u] >= n2) {            // cycle walking: rare, lanes on their own
            uint32_t L, R;
            dom.split(x2[u] >> 1, L, R);
            x2[u] = inverse2(2u * L, 2u * R);
          }
      }
#pragma unroll
      for (int u = 0; u < NI; ++u) {
        uint32_t q = mulhi32(x2[u], magic2);
        if ((q + 1u) * B2 <= x2[u]) ++q;
        const uint32_t key = live[u] ? q : 0xffffffffu;          // dead lanes form their own group and write nothing
        const unsigned same = __match_any_sync(FULL, key);
        const unsigned below = __popc(same & lt);
        int old = 0;
        if (live[u]) {
          old = s_wh[warp * 64 + q];                              // the warp's own counters
          s_sr[base + 32 * u + lane] = (unsigned short)(q | ((uint32_t)(old + below) << sb));
        }
        __syncwarp();
        if (live[u] && below == 0) s_wh[warp * 64 + q] = old + __popc(same);
        __syncwarp();
      }
    }
    __syncthreads();
    // ---- warp 0: exclusive scan of the counts in (step, warp) order (entry e = step * NW + warp, C per lane);
    // the other warps build the next row's round tables meanwhile
    if (warp == 0) {
      const int T = spe * NW, C = (T + 31) / 32;
      const int e0 = lane * C;
      int sum = 0;
      for (int c = 0; c < C; ++c) {
        const int e = e0 + c;
        if (e < T) sum += s_wh[(e % NW) * 64 + e / NW];
      }
      int inc = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(FULL, inc, o);
        if (lane >= o) inc += t;
      }
      int run = inc - sum;
      for (int c = 0; c < C; ++c) {
        const int e = e0 + c;
        if (e < T) {
          int* const p = &s_wh[(e % NW) * 64 + e / NW];
          const int v = *p;
          *p = run;
          if (e % NW == 0) off[e / NW] = run;
          run += v;
        }
      }
      if (lane == 0) off[spe] = m;
    } else {
      const int rn = r + gridDim.y;
      if (rn < hp.owner_sched_rows && e_first + rn < epochs)
        build_tables(e_first + rn, s_tab + ((it + 1) & 1) * 4 * tab_bytes, tid - 32, kSchedThreads - 32);
    }
    __syncthreads();
    // ---- pass 2: position = start of (step, warp) + rank; then the warp clears its counters for the next row
    for (int sl = w0 + lane; sl < w1; sl += 32) {
      const uint32_t pk = s_sr[sl];
      out[s_wh[warp * 64 + (pk & qmask)] + (pk >> sb)] = (unsigned short)sl;
    }
    __syncwarp();
    s_wh[warp * 64 + lane] = 0;
    s_wh[warp * 64 + 32 + lane] = 0;
    __syncwarp();
  }
}

// ---------------------------------------------------------------- the training kernel
// The loop below is issue-bound (ncu: ~50 % issue-slot utilisation, profiles/): launch-uniform array bases,
// 32-bit shared-memory indexing, packed cache records and compile-time CACHED keep its instruction count down.
// LONGLIST: the launch's owner_cap_list is below owner_cap_slots, so a batch list may have to be read from the
// schedule table in global memory (generic loads); false keeps every list access a shared-memory load.
template <int D, bool CACHED, bool LONGLIST>
__global__ void __launch_bounds__(kOwnThreads, 1)
mf_owner_kernel(const ure_mf_shard_t* __restrict__ shards, int K, ure_mf_hparams_t hp, int epochs,
                long long step_begin, long long step_end, OwnerWs* ws) {
  constexpr int CH = D / 4;                // float4 chunks of a row
  // lanes per interaction and chunks per lane: one chunk per lane up to d=32; wide rows give every lane V=4 chunks
  // (chunk gl + v*G: a load instruction of the group still covers G*16 contiguous bytes), which divides the
  // shuffle reductions and the per-interaction bookkeeping (the loop is issue-bound) by four.
  constexpr int V = D >= 64 ? 4 : 1;
  constexpr int G = CH / V;                // lanes per interaction
  constexpr int GPW = 32 / G;              // lane groups per warp
  constexpr int QB = V == 4 ? 2 : 4;       // interactions a group handles per wave (QB*V gathers in flight per lane)
  constexpr int WAVE = GPW * QB;           // interactions per warp and wave
  constexpr int NW = kOwnWarps;
  constexpr int RS = 2 * D;                // row stride in floats: [w | momentum, pre-scaled: mu*buf + wd*w]
  constexpr unsigned FULL = 0xffffffffu;
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ PlanScratch s_ps;
  __shared__ Plan s_pl;
  __shared__ ure_mf_shard_t s_sh;
  __shared__ float s_wsse[NW];
  __shared__ int s_total;                  // entries of the batch list in s_list

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, gl = lane % G, gw = lane / G;
  if (hp.owner_plan && ld_acquire_u32(reinterpret_cast<const unsigned*>(&ws->error)) == 2u) return;   // uniform over the grid: the pre-pass found the remembered capacities too small
  make_plan(shards, K, blockIdx.x, gridDim.x, s_pl, s_ps);
  if (tid == 0) s_sh = shards[s_pl.shard];
  __syncthreads();
  const ure_mf_shard_t& sh = s_sh;
  const int ru0 = s_pl.ru0, ri0 = s_pl.ri0, mU = s_pl.mU;
  const int rowsU = s_pl.ru1 - ru0, rows = rowsU + (s_pl.ri1 - ri0);
  const int m = mU + s_pl.mI;
  const int B = hp.batch;
  const int n = sh.n;
  const int spe = (n + B - 1) / B;
  const long long t_end = spe > 0 ? min(step_end, (long long)spe * epochs) : step_begin;
  if (t_end <= step_begin) return;         // the whole shard (all of its CTAs) has nothing to do

  // ---- shared-memory carve-up: bases depend on kernel parameters only
  const int cap = hp.owner_cap_slots;      // multiple of 16, >= m
  const int lcap = hp.owner_cap_list;      // multiple of 16: batch lists up to this length are staged in s_list
  float* const s_bnd = reinterpret_cast<float*>(dyn);                       // [2*NW][D] boundary-row partial sums
  unsigned short* const s_list = reinterpret_cast<unsigned short*>(s_bnd + 2 * NW * D);   // [lcap] slots of the batch
  // packed records: CACHED: of every owned slot [cap]; else of the entries of the staged batch list [lcap]
  uint2* const s_rec = reinterpret_cast<uint2*>(s_list + lcap);
  float* const s_w = reinterpret_cast<float*>(s_rec + (CACHED ? cap : lcap));   // row r: s_w + r*RS
  float* const s_b = s_w + D;              // gradients are summed straight into the pre-scaled momentum
  int* const s_bidx = reinterpret_cast<int*>(s_w + hp.owner_cap_rows * RS);   // [rows] first boundary record, or INT_MAX
  int* const s_blast = s_bidx + hp.owner_cap_rows;                            // [rows] last boundary record, or -1

  const int4* const recU = reinterpret_cast<const int4*>(sh.inter_u + s_pl.su0);           // slot sl < mU
  const int4* const recI = reinterpret_cast<const int4*>(sh.inter_i + s_pl.si0) - mU;      // slot sl >= mU
  auto pack_rec = [&](const int4& rec, bool it) {       // {other | own row << kOtherBits, rating}
    const unsigned row = (unsigned)(it ? rec.y - ri0 + rowsU : rec.x - ru0);
    return make_uint2((unsigned)(it ? rec.x : rec.y) | (row << kOtherBits), (unsigned)rec.z);
  };
  auto load_rec = [&](int sl) { return __ldg((sl >= mU ? recI : recU) + sl); };
  const int offF = (int)(s_bnd - s_b) + 2 * warp * D, offL = offF + D;      // float offsets relative to s_b

  // the CTA's part of the schedule (ure_mf_owner_schedule): row of the shard's epoch, run of the step
  const int sched_e0 = (int)(hp.owner_sched_step0 / spe);
  const unsigned short* const sched = hp.owner_sched + s_pl.slot_base;
  const int* const sched_off = hp.owner_sched_off + (long long)blockIdx.x * (hp.owner_spe_cap + 1);
  const long long off_row = (long long)gridDim.x * (hp.owner_spe_cap + 1);
  // where the batch list of (epoch ep, step kk) lives: false = outside the scheduled window
  auto find_list = [&](int ep, int kk, const unsigned short*& src, int& len) {
    const int row = ep - sched_e0;
    src = sched;
    len = 0;
    if (row < 0 || row >= hp.owner_sched_rows) return false;
    const int* o = sched_off + row * off_row + kk;
    const int a = __ldcg(o), b = __ldcg(o + 1);
    src = sched + row * hp.owner_sched_stride + a;
    len = b - a;
    return true;
  };
  // The list of step t+1 is fetched into registers at the START of step t (its address was looked up in the
  // barrier shadow of step t-1) and stored to s_list in the shadow of step t: no global latency in the shadow.
  // Without the record cache the records of the staged list travel with it: loaded into registers when the
  // waves are done (the list entries have arrived by then), stored next to the list in the shadow.
  constexpr int PF = 6;                    // register entries per thread; longer lists copy the rest directly
  constexpr int PFR = 2;                   // ... of which this many also carry their record
  unsigned short pf[PF];
  int4 pr[PFR];
  const unsigned short* nx_src = sched;    // list of the NEXT step
  int nx_len = 0;
  bool nx_ok = true;
  const unsigned short* cur_src = sched;   // list of THIS step in the schedule table (read there when > lcap)

  // ---- prologue: owned rows -> shared memory, record cache, first batch list
  for (int x = tid; x < rows * CH; x += kOwnThreads) {
    const int r = x / CH, c = x % CH;
    const bool it = r >= rowsU;
    const size_t go = (size_t)(it ? ri0 + (r - rowsU) : ru0 + r) * D + 4 * c;
    const float4 w = ld_cg_f4((it ? sh.Q : sh.P) + go);
    float4 b = ld_cg_f4((it ? sh.bufQ : sh.bufP) + go);
    // pre-scaled momentum: mu*buf + wd*w, what torch SGD adds the batch gradient to (buf = mu*buf + (g + wd*w))
    b.x = fmaf(hp.momentum, b.x, hp.weight_decay * w.x); b.y = fmaf(hp.momentum, b.y, hp.weight_decay * w.y);
    b.z = fmaf(hp.momentum, b.z, hp.weight_decay * w.z); b.w = fmaf(hp.momentum, b.w, hp.weight_decay * w.w);
    *reinterpret_cast<float4*>(s_w + r * RS + 4 * c) = w;
    *reinterpret_cast<float4*>(s_b + r * RS + 4 * c) = b;
  }
  for (int x = tid; x < 2 * NW * CH; x += kOwnThreads)
    *reinterpret_cast<float4*>(s_bnd + 4 * x) = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int r = tid; r < rows; r += kOwnThreads) { s_bidx[r] = 0x7fffffff; s_blast[r] = -1; }
  if (CACHED)
    for (int sl = tid; sl < m; sl += kOwnThreads) s_rec[sl] = pack_rec(__ldg((sl >= mU ? recI : recU) + sl), sl >= mU);
  int e = (int)(step_begin / spe), k = (int)(step_begin % spe);
  bool in_window;
  {
    const unsigned short* src;
    int len;
    in_window = find_list(e, k, src, len);
    cur_src = src;
    if (len <= lcap)
      for (int x = tid; x < len; x += kOwnThreads) {
        const int sl = __ldcg(src + x);
        s_list[x] = (unsigned short)sl;
        if (!CACHED) s_rec[x] = pack_rec(load_rec(sl), sl >= mU);
      }
    if (tid == 0) s_total = len;
    if (step_begin + 1 < t_end) nx_ok = find_list(k + 1 == spe ? e + 1 : e, k + 1 == spe ? 0 : k + 1, nx_src, nx_len);
  }
  __syncthreads();

  auto lr_of = [&](int epoch) {
    double lr = (double)hp.lr0;
    for (int q = epoch / hp.lr_step; q > 0; --q) lr *= (double)hp.lr_decay;
    return (float)lr;
  };
  float nlr = -lr_of(e);
  const float wd = hp.weight_decay, mu = hp.momentum;
  unsigned* const counter = &ws->bar[s_pl.shard][0];
  const unsigned n_cta = (unsigned)s_pl.c;
  unsigned bar_target = 0;
  double epoch_sse = 0.0;                  // thread 0 only
  long long* const trace = ws->trace;
  const int trace_steps = ws->trace_steps;
#define URE_STAMP(PH)                                                               \
  if (trace && tid == 32 && (t - step_begin) < trace_steps)                        \
    trace[((t - step_begin) * gridDim.x + blockIdx.x) * 6 + (PH)] = clock64();

  for (long long t = step_begin; t < t_end; ++t) {
    if (!in_window) {                      // uniform over the shard's CTAs: all of them stop at the same step
      if (tid == 0) atomicMax(&ws->error, 1);
      break;
    }
    const bool rd = (t - step_begin) & 1;
    const float* const Pr = rd ? sh.gP : sh.P;
    const float* const Qr = rd ? sh.gQ : sh.Q;
    float sse_l = 0.f;
    const int total = s_total;
    const bool staged = !LONGLIST || total <= lcap;                          // uniform over the CTA
    const unsigned short* const lst = staged ? s_list : cur_src;
    const bool last_step = t + 1 == t_end;
    auto rec_at = [&](int pos) {           // packed record of list entry pos
      if (CACHED) return s_rec[lst[pos]];
      if (staged) return s_rec[pos];
      const int sl = lst[pos];
      return pack_rec(load_rec(sl), sl >= mU);
    };
    URE_STAMP(0)
#pragma unroll
    for (int i = 0; i < PF; ++i) {         // next step's list on its way into registers
      const int x = tid + i * kOwnThreads;
      pf[i] = x < nx_len ? __ldcg(nx_src + x) : (unsigned short)0;
    }

    // -------------------------------------------------------------- waves: this warp's contiguous share of the
    // sorted batch list.  Only the first and the last row of the share can be shared with other warps: their
    // partial sums go to the warp's two boundary records, everything else straight to the row's accumulator
    // (plain read-modify-write: within the warp, flushes of one row are at different program points with a
    // __syncwarp between them).
    const int n_waves = (total + WAVE - 1) / WAVE;
    const int wv0 = warp * (n_waves / NW) + min(warp, n_waves % NW);
    const int wv1 = wv0 + n_waves / NW + (warp < n_waves % NW ? 1 : 0);
    const int ent1 = min(total, wv1 * WAVE);
    int rowF = -1, rowL = -1;
    if (wv0 < wv1) {
      rowF = (int)(rec_at(wv0 * WAVE).x >> kOtherBits);
      rowL = (int)(rec_at(ent1 - 1).x >> kOtherBits);
    }
    if (lane == 0) {
      if (rowF >= 0) {
        atomicMin(&s_bidx[rowF], 2 * warp); atomicMax(&s_blast[rowF], 2 * warp);
        atomicMin(&s_bidx[rowL], 2 * warp + 1); atomicMax(&s_blast[rowL], 2 * warp + 1);
      }
    }
    auto flush = [&](int row, const float4 (&a)[V]) {
      if (row >= 0) {
        float* const base = s_b + (row == rowF ? offF : row == rowL ? offL : row * RS) + 4 * gl;
#pragma unroll
        for (int v = 0; v < V; ++v) {
          float4* gp = reinterpret_cast<float4*>(base + 4 * v * G);
          float4 x = *gp;
          x.x += a[v].x; x.y += a[v].y; x.z += a[v].z; x.w += a[v].w;
          *gp = x;
        }
      }
    };
    for (int wv = wv0; wv < wv1; ++wv) {
      const int ent0 = wv * WAVE + gw * QB;
      int row[QB];
      float rat[QB];
      float4 o4[QB][V];
#pragma unroll
      for (int q = 0; q < QB; ++q) {       // branch-free: entries past the end re-read the last one, weight 0
        const uint2 rec = rec_at(min(ent0 + q, ent1 - 1));
        const bool ok = ent0 + q < ent1;
        const int r = (int)(rec.x >> kOtherBits);
        row[q] = ok ? r : -1;
        rat[q] = __uint_as_float(rec.y);
        // L1-allocating load: a CTA re-reads popular rows within a step; the acquire load that ends every
        // barrier invalidates L1 (CCTL.IVALL), so no line survives into the step that rewrites its buffer
        const float* const src = (r >= rowsU ? Pr : Qr) + (size_t)(rec.x & ((1u << kOtherBits) - 1u)) * D + 4 * gl;
#pragma unroll
        for (int v = 0; v < V; ++v) o4[q][v] = __ldca(reinterpret_cast<const float4*>(src + 4 * v * G));
      }
      int key;
      float4 acc[V];
      if constexpr (V == 4) {
        // wide rows, two interactions per group: both chains run side by side (four partial dot sums each, the
        // gathered row scaled in place into its gradient contribution); the row change inside the group is
        // resolved after both are done
        static_assert(V != 4 || QB == 2, "the wide-row wave handles two interactions per group");
        float dot[QB];
#pragma unroll
        for (int q = 0; q < QB; ++q) {
          const float* const wrow = s_w + max(row[q], 0) * RS + 4 * gl;
          float p[V];
#pragma unroll
          for (int v = 0; v < V; ++v) {
            const float4 w = *reinterpret_cast<const float4*>(wrow + 4 * v * G);
            p[v] = w.x * o4[q][v].x;
            p[v] = fmaf(w.y, o4[q][v].y, p[v]);
            p[v] = fmaf(w.z, o4[q][v].z, p[v]);
            p[v] = fmaf(w.w, o4[q][v].w, p[v]);
          }
          dot[q] = (p[0] + p[1]) + (p[2] + p[3]);
        }
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) {
#pragma unroll
          for (int q = 0; q < QB; ++q) dot[q] += __shfl_xor_sync(FULL, dot[q], o);
        }
#pragma unroll
        for (int q = 0; q < QB; ++q) {
          const float err = row[q] >= 0 ? dot[q] - rat[q] : 0.f;
          const float ge = 2.f * err;
          if (row[q] < rowsU) sse_l = fmaf(err, err, sse_l);    // every lane of the group: divided by G below
#pragma unroll
          for (int v = 0; v < V; ++v) {
            o4[q][v].x *= ge; o4[q][v].y *= ge; o4[q][v].z *= ge; o4[q][v].w *= ge;
          }
        }
        key = row[1];
        if (row[0] == row[1]) {
#pragma unroll
          for (int v = 0; v < V; ++v) {
            acc[v].x = o4[0][v].x + o4[1][v].x; acc[v].y = o4[0][v].y + o4[1][v].y;
            acc[v].z = o4[0][v].z + o4[1][v].z; acc[v].w = o4[0][v].w + o4[1][v].w;
          }
        } else {
          flush(row[0], o4[0]);
#pragma unroll
          for (int v = 0; v < V; ++v) acc[v] = o4[1][v];
        }
      } else {
      key = -1;
#pragma unroll
      for (int v = 0; v < V; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int q = 0; q < QB; ++q) {
        const float* const wrow = s_w + max(row[q], 0) * RS + 4 * gl;
        float dot = 0.f;
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const float4 w = *reinterpret_cast<const float4*>(wrow + 4 * v * G);
          dot = v == 0 ? w.x * o4[q][v].x : fmaf(w.x, o4[q][v].x, dot);
          dot = fmaf(w.y, o4[q][v].y, dot);
          dot = fmaf(w.z, o4[q][v].z, dot);
          dot = fmaf(w.w, o4[q][v].w, dot);
        }
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) dot += __shfl_xor_sync(FULL, dot, o);
        const float err = row[q] >= 0 ? dot - rat[q] : 0.f;
        const float ge = 2.f * err;
        if (row[q] < rowsU) sse_l = fmaf(err, err, sse_l);      // every lane of the group: divided by G below
        if (q > 0 && row[q] != key) {      // the row changes inside the group: the finished run goes out
          flush(key, acc);
#pragma unroll
          for (int v = 0; v < V; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        key = row[q];
#pragma unroll
        for (int v = 0; v < V; ++v) {
          acc[v].x = fmaf(ge, o4[q][v].x, acc[v].x); acc[v].y = fmaf(ge, o4[q][v].y, acc[v].y);
          acc[v].z = fmaf(ge, o4[q][v].z, acc[v].z); acc[v].w = fmaf(ge, o4[q][v].w, acc[v].w);
        }
      }
      }
      // segmented reduction of the groups' trailing runs (the list is sorted, equal rows are adjacent).  Wide rows
      // (V = 4: sixteen values per lane and step of the reduction) skip it when no two neighbouring groups end in
      // the same row -- the usual case when a step brings about one interaction per owned row.
      const int kprev = __shfl_up_sync(FULL, key, G);
      const bool shared_runs = V == 1 || __any_sync(FULL, gw > 0 && kprev == key);
      if (shared_runs) {
#pragma unroll
      for (int o = 1; o < GPW; o <<= 1) {
        const int k2 = __shfl_down_sync(FULL, key, o * G);
        const bool take = gw + o < GPW && k2 == key;
#pragma unroll
        for (int v = 0; v < V; ++v) {
          float4 a2;
          a2.x = __shfl_down_sync(FULL, acc[v].x, o * G); a2.y = __shfl_down_sync(FULL, acc[v].y, o * G);
          a2.z = __shfl_down_sync(FULL, acc[v].z, o * G); a2.w = __shfl_down_sync(FULL, acc[v].w, o * G);
          if (take) { acc[v].x += a2.x; acc[v].y += a2.y; acc[v].z += a2.z; acc[v].w += a2.w; }
        }
      }
      }
      __syncwarp();                        // the in-group flushes above are visible to the head flushes below
      if (gw == 0 || kprev != key) flush(key, acc);
      __syncwarp();
    }
    sse_l = warp_sum(sse_l);
    if (lane == 0) s_wsse[warp] = sse_l * (1.f / G);
    const int stage = (t + 1 < t_end && nx_len <= lcap) ? nx_len : 0;   // a list longer than s_list stays in the table
    if (!CACHED) {
#pragma unroll
      for (int i = 0; i < PFR; ++i) {      // the next list's records: in flight during the row sweep
        const int x = tid + i * kOwnThreads;
        pr[i] = load_rec(x < stage ? (int)pf[i] : 0);
      }
    }
    URE_STAMP(1)
    __syncthreads();
    URE_STAMP(2)

    // ------------------------------------------------------------ SGD update of every owned row, publication
    {
      float* const Pw = rd ? sh.P : sh.gP;
      float* const Qw = rd ? sh.Q : sh.gQ;
#pragma unroll 4
      for (int x = tid; x < rows * CH; x += kOwnThreads) {
        const int r = x / CH, c = x % CH;
        float4* wp = reinterpret_cast<float4*>(s_w + r * RS + 4 * c);
        float4* bp = wp + D / 4;
        float4 w = *wp, b = *bp;             // b: mu*buf + wd*w + the gradients flushed by the waves
        // boundary rows: the partial sums of the warps that shared the row (adjacent records, in list order)
        // (records first..last: all of this row or of warps without entries, whose records are zero)
        const int bi = s_bidx[r];
        if (bi != 0x7fffffff) {
          const int bl = s_blast[r];
          for (int j = bi; j <= bl; ++j) {
            float4* rp = reinterpret_cast<float4*>(s_bnd + j * D + 4 * c);
            const float4 v = *rp;
            b.x += v.x; b.y += v.y; b.z += v.z; b.w += v.w;
            *rp = make_float4(0.f, 0.f, 0.f, 0.f);
          }
          __syncwarp(__activemask());
          if (c == 0) { s_bidx[r] = 0x7fffffff; s_blast[r] = -1; }
        }
        // torch SGD: buf = mu*buf + (g + wd*w); w = w + (-lr)*buf -- b is the new buf; the next step's pre-scaled
        // momentum mu*b + wd*w replaces it, except after the launch's last step (the epilogue stores buf itself)
        w.x = fmaf(nlr, b.x, w.x); w.y = fmaf(nlr, b.y, w.y); w.z = fmaf(nlr, b.z, w.z); w.w = fmaf(nlr, b.w, w.w);
        *wp = w;
        if (!last_step) {
          b.x = fmaf(mu, b.x, wd * w.x); b.y = fmaf(mu, b.y, wd * w.y);
          b.z = fmaf(mu, b.z, wd * w.z); b.w = fmaf(mu, b.w, wd * w.w);
        }
        *bp = b;
        const bool it = r >= rowsU;
        st_cg_f4((it ? Qw : Pw) + (size_t)(it ? ri0 + (r - rowsU) : ru0 + r) * D + 4 * c, w);
      }
    }
    __syncthreads();                       // every row of this CTA is updated and published
    URE_STAMP(3)

    // ------------------------------------------------------------ barrier among the shard's CTAs
    if (tid == 0) asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
    __syncwarp();
    bar_target += n_cta;
    const bool last_of_epoch = k + 1 == spe;
    // in the barrier's shadow: the NEXT step's list goes to shared memory, the one after is looked up
    if (t + 1 < t_end) {
      in_window = nx_ok;
      cur_src = nx_src;
#pragma unroll
      for (int i = 0; i < PF; ++i) {
        const int x = tid + i * kOwnThreads;
        if (x < stage) {
          s_list[x] = pf[i];
          if (!CACHED) s_rec[x] = pack_rec(i < PFR ? pr[i < PFR ? i : 0] : load_rec(pf[i]), pf[i] >= mU);
        }
      }
      for (int x = tid + PF * kOwnThreads; x < stage; x += kOwnThreads) {
        const int sl = __ldcg(nx_src + x);
        s_list[x] = (unsigned short)sl;
        if (!CACHED) s_rec[x] = pack_rec(load_rec(sl), sl >= mU);
      }
      if (tid == 0) s_total = nx_len;
      if (t + 2 < t_end) {
        int e2 = last_of_epoch ? e + 1 : e, k2 = last_of_epoch ? 0 : k + 1;      // step t+1 ...
        if (k2 + 1 == spe) { ++e2; k2 = 0; } else ++k2;                            // ... and t+2
        nx_ok = find_list(e2, k2, nx_src, nx_len);
      }
    }
    URE_STAMP(4)
    if (tid == 0) {
      float v = 0.f;
      for (int w = 0; w < NW; ++w) v += s_wsse[w];
      epoch_sse += (double)v;
      if (last_of_epoch || t + 1 == t_end || !in_window) {
        if (epoch_sse != 0.0) atomicAdd(sh.sse + e, epoch_sse);
        epoch_sse = 0.0;
      }
      while (ld_acquire_u32(counter) < bar_target) {}
    }
    __syncthreads();
    URE_STAMP(5)
    if (last_of_epoch) { ++e; k = 0; nlr = -lr_of(e); }
    else ++k;
  }
#undef URE_STAMP

  // ---- epilogue: the owned rows go back to P/Q (whatever the parity), momentum to bufP/bufQ, and the
  // alternate weight buffer gP/gQ is returned zeroed (the DENSE schedule's contract for its gradient scratch)
  for (int x = tid; x < rows * CH; x += kOwnThreads) {
    const int r = x / CH, c = x % CH;
    const bool it = r >= rowsU;
    const size_t go = (size_t)(it ? ri0 + (r - rowsU) : ru0 + r) * D + 4 * c;
    st_cg_f4((it ? sh.Q : sh.P) + go, *reinterpret_cast<const float4*>(s_w + r * RS + 4 * c));
    st_cg_f4((it ? sh.bufQ : sh.bufP) + go, *reinterpret_cast<const float4*>(s_b + r * RS + 4 * c));
    st_cg_f4((it ? sh.gQ : sh.gP) + go, make_float4(0.f, 0.f, 0.f, 0.f));
  }
}

int max_dyn_smem(int* out) {
  int dev = 0, v = 0;
  URE_CUDA(cudaGetDevice(&dev));
  URE_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  *out = v - 8 * 1024;                     // minus the kernel's static shared memory (plan scratch, descriptor)
  return 0;
}

template <int D>
int launch_owner(const ure_mf_shard_t* d_shards, int K, const ure_mf_hparams_t& hp, int epochs, long long s0,
                 long long s1, OwnerWs* ws, int smem, bool cached, cudaStream_t st) {
  const bool longlist = hp.owner_cap_list < hp.owner_cap_slots;
  auto kern = cached ? mf_owner_kernel<D, true, false>
                     : longlist ? mf_owner_kernel<D, false, true> : mf_owner_kernel<D, false, false>;
  URE_REQUIRE(!(cached && longlist), URE_EINVAL, "ure_mf_train(owner): the record cache needs owner_cap_list == owner_cap_slots");
  URE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  URE_CUDA(cudaMemsetAsync(ws->bar, 0, sizeof(ws->bar), st));
  void* args[] = {(void*)&d_shards, (void*)&K, (void*)&hp, (void*)&epochs, (void*)&s0, (void*)&s1, (void*)&ws};
  URE_CUDA(cudaLaunchCooperativeKernel((void*)kern, dim3(num_sms()), dim3(kOwnThreads), args, (size_t)smem, st));
  return 0;
}

}  // namespace

int64_t mf_owner_workspace_bytes() { return (int64_t)sizeof(OwnerWs); }
int mf_owner_trace(void* d_workspace, long long* d_trace, int steps, cudaStream_t st) {
  auto* ws = static_cast<OwnerWs*>(d_workspace);
  URE_CUDA(cudaMemcpyAsync(&ws->trace, &d_trace, sizeof(d_trace), cudaMemcpyHostToDevice, st));
  URE_CUDA(cudaMemcpyAsync(&ws->trace_steps, &steps, sizeof(int), cudaMemcpyHostToDevice, st));
  URE_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// called by ure_mf_train when hparams.mode == URE_MF_OWNER; the capacities in hparams are the plan's maxima the
// caller read back after ure_mf_owner_prepare (the library never synchronises)
int mf_train_owner(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* hp, int epochs,
                   long long step_begin, long long step_end, void* d_workspace, cudaStream_t st) {
  URE_REQUIRE(n_shards <= num_sms(), URE_EUNSUPPORTED,
              "ure_mf_train(owner): %d shards need at least as many SMs (%d)", n_shards, num_sms());
  URE_REQUIRE(hp->owner_cap_rows > 0 && hp->owner_cap_slots >= 0 && hp->owner_cap_slots % 16 == 0, URE_EINVAL,
              "ure_mf_train(owner): hparams.owner_cap_rows / owner_cap_slots must carry the plan of "
              "ure_mf_owner_prepare (slots rounded up to a multiple of 16)");
  URE_REQUIRE(hp->owner_cap_slots <= 65520 && hp->owner_cap_rows < (1 << (32 - kOtherBits)), URE_EUNSUPPORTED,
              "ure_mf_train(owner): %d interactions / %d rows per CTA exceed the 16-bit slot / 12-bit row fields",
              hp->owner_cap_slots, hp->owner_cap_rows);
  URE_REQUIRE(hp->owner_sched && hp->owner_sched_off && hp->owner_sched_rows > 0 && hp->owner_sched_step0 <= step_begin,
              URE_EINVAL, "ure_mf_train(owner): no schedule for step %lld (ure_mf_owner_schedule first)", step_begin);
  URE_REQUIRE(hp->owner_cap_list >= 16 && hp->owner_cap_list % 16 == 0 && hp->owner_cap_list <= hp->owner_cap_slots,
              URE_EINVAL, "ure_mf_train(owner): hparams.owner_cap_list=%d must be a multiple of 16 in [16, owner_cap_slots]",
              hp->owner_cap_list);
  const bool cached = (hp->owner_flags & 1) != 0;
  const long long need = owner_smem_bytes(hp->d, hp->owner_cap_rows, hp->owner_cap_slots, hp->owner_cap_list, cached);
  int avail = 0;
  if (int rc = max_dyn_smem(&avail)) return rc;
  URE_REQUIRE(need <= avail, URE_EUNSUPPORTED,
              "ure_mf_train(owner): the plan needs %lld bytes of shared memory per CTA, %d available -- use the "
              "dense or lazy schedule for this problem size", need, avail);
  if (step_end <= step_begin) return 0;
  auto* ws = static_cast<OwnerWs*>(d_workspace);
  const int smem = (int)need;
  switch (hp->d) {
    case 8: return launch_owner<8>(d_shards, n_shards, *hp, epochs, step_begin, step_end, ws, smem, cached, st);
    case 16: return launch_owner<16>(d_shards, n_shards, *hp, epochs, step_begin, step_end, ws, smem, cached, st);
    case 32: return launch_owner<32>(d_shards, n_shards, *hp, epochs, step_begin, step_end, ws, smem, cached, st);
    case 64: return launch_owner<64>(d_shards, n_shards, *hp, epochs, step_begin, step_end, ws, smem, cached, st);
    case 128: return launch_owner<128>(d_shards, n_shards, *hp, epochs, step_begin, step_end, ws, smem, cached, st);
    default:
      set_error("ure_mf_train(owner): d=%d not in {8,16,32,64,128}", hp->d);
      return URE_EUNSUPPORTED;
  }
}

}  // namespace ure

extern "C" int64_t ure_mf_owner_smem_bytes(int d, int cap_rows, int cap_slots, int cap_list, int spe_cap, int flags) {
  const long long a = ure::owner_smem_bytes(d, cap_rows, cap_slots, cap_list, (flags & 1) != 0);
  const long long b = ure::schedule_smem_bytes(cap_slots, spe_cap, (flags & 2) == 0);
  return a > b ? a : b;
}

extern "C" int ure_mf_owner_schedule(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp,
                                     int epochs, int64_t step0, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_shards && h_hp && h_hp->owner_sched && h_hp->owner_sched_off, URE_EINVAL,
              "ure_mf_owner_schedule: null argument");
  URE_REQUIRE(h_hp->owner_sched_rows >= 1 && h_hp->owner_spe_cap >= 1 && h_hp->owner_spe_cap <= kMaxSpe &&
                  h_hp->owner_cap_slots % 16 == 0 && h_hp->owner_cap_slots <= 65520,
              URE_EUNSUPPORTED, "ure_mf_owner_schedule: rows=%d spe_cap=%d cap_slots=%d outside the supported range",
              h_hp->owner_sched_rows, h_hp->owner_spe_cap, h_hp->owner_cap_slots);
  int avail = 0;
  if (int rc = max_dyn_smem(&avail)) return rc;
  ure_mf_hparams_t hp = *h_hp;
  hp.owner_sched_step0 = step0;
  const int ny = h_hp->owner_sched_rows < 4 ? h_hp->owner_sched_rows : 4;    // 2 blocks per SM, 2 rounds
  const bool cache_j = (h_hp->owner_flags & 2) == 0;
  // round-function tables of the visiting order when they fit next to the rest (a, b ~ sqrt(n) entries each)
  int tab_cap = 0;
  if (h_hp->owner_max_n > 1) {
    FeistelDomain dom;
    dom.init((uint32_t)h_hp->owner_max_n);             // a >= b and a grows with n: the largest shard sizes the tables
    const int cap = (int)((dom.a > dom.b ? dom.a : dom.b) + 2 + 7) / 8 * 8;
    if (cap <= kTabMaxHalf && schedule_smem_bytes(h_hp->owner_cap_slots, h_hp->owner_spe_cap, cache_j, cap) <= avail) tab_cap = cap;
  }
  // short epochs with round tables: the tight kernel (two CTAs per SM, one wave)
  int sb = 1;
  while ((1 << sb) < h_hp->owner_spe_cap) ++sb;
  const int per = (((h_hp->owner_cap_slots + kSchedWarps - 1) / kSchedWarps) + 31) & ~31;
  const long long need_t = schedule_tab_smem_bytes(h_hp->owner_cap_slots, tab_cap);
  if (tab_cap > 0 && h_hp->owner_spe_cap <= 64 && per < (1 << (16 - sb)) && need_t <= avail) {
    URE_CUDA(cudaFuncSetAttribute(owner_schedule_tab_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need_t));
    const int ny2 = h_hp->owner_sched_rows < 2 ? h_hp->owner_sched_rows : 2;
    owner_schedule_tab_kernel<<<dim3(num_sms(), ny2), kSchedThreads, (size_t)need_t, static_cast<cudaStream_t>(stream)>>>(
        d_shards, n_shards, hp, epochs, step0, tab_cap, sb);
    URE_CUDA(cudaGetLastError());
    return 0;
  }
  const long long need = schedule_smem_bytes(h_hp->owner_cap_slots, h_hp->owner_spe_cap, cache_j, tab_cap);
  URE_REQUIRE(need <= avail, URE_EUNSUPPORTED, "ure_mf_owner_schedule: %lld bytes of shared memory needed, %d available",
              need, avail);
  URE_CUDA(cudaFuncSetAttribute(owner_schedule_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
  owner_schedule_kernel<<<dim3(num_sms(), ny), kSchedThreads, (size_t)need, static_cast<cudaStream_t>(stream)>>>(
      d_shards, n_shards, hp, epochs, step0, tab_cap);
  URE_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------- per-user segments of a test set (baseTest)
// The host dict of method/utils.py:151-161 groups the test rows by user, a user's rows in file order.  Here: the
// same stable radix sort the owner set-up uses (user side only) on the test records, CSR offsets by user id.
namespace ure {
namespace {
__global__ void seg_count_kernel(const ure_inter_t* __restrict__ inter, long long n, int n_user, int32_t* off_u,
                                 int* __restrict__ bad) {
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x) {
    const int u = inter[j].user;
    if (u < 0 || u >= n_user) { *bad = 1; continue; }
    atomicAdd(off_u + u + 1, 1);
  }
}
__global__ void seg_extract_kernel(const ure_inter_t* __restrict__ sorted, long long n, const int32_t* __restrict__ off_u,
                                   int n_user, int32_t* __restrict__ order, long long* __restrict__ seg) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) order[j] = sorted[j].pad;
  for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u <= n_user; u += stride) seg[u] = off_u[u];
}
inline int64_t seg_align(int64_t x) { return (x + 255) / 256 * 256; }
}  // namespace
}  // namespace ure

extern "C" int64_t ure_user_segments_scratch_bytes(int64_t n, int n_user) {
  using namespace ure;
  return 256 + seg_align(((int64_t)n_user + 2) * 4) + 2 * seg_align(n * 16) + seg_align(256ll * kRadixBlocks * 4) + 256;
}

extern "C" int ure_user_segments(const ure_inter_t* d_inter, int64_t n, int n_user, int32_t* d_order, int64_t* d_seg,
                                 void* d_scratch, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_inter && d_order && d_seg && d_scratch && n > 0 && n_user > 0 && n < (1ll << 31), URE_EINVAL,
              "ure_user_segments: bad argument (n=%lld, n_user=%d)", (long long)n, n_user);
  auto st = static_cast<cudaStream_t>(stream);
  char* base = static_cast<char*>(d_scratch);
  auto* d_desc = reinterpret_cast<ure_mf_shard_t*>(base);
  auto* off_u = reinterpret_cast<int32_t*>(base + 256);
  char* p = base + 256 + seg_align(((int64_t)n_user + 2) * 4);
  auto* sorted = reinterpret_cast<ure_inter_t*>(p); p += seg_align(n * 16);
  auto* tmp = reinterpret_cast<ure_inter_t*>(p); p += seg_align(n * 16);
  auto* hist = reinterpret_cast<int*>(p); p += seg_align(256ll * kRadixBlocks * 4);
  int* bad = reinterpret_cast<int*>(p);
  ure_mf_shard_t h;
  memset(&h, 0, sizeof(h));
  h.inter = d_inter; h.inter_u = sorted; h.tmp_u = tmp; h.off_u = off_u; h.n = (int32_t)n; h.n_user = n_user;
  URE_CUDA(cudaMemcpyAsync(d_desc, &h, sizeof(h), cudaMemcpyHostToDevice, st));
  URE_CUDA(cudaMemsetAsync(off_u, 0, ((size_t)n_user + 2) * 4, st));
  URE_CUDA(cudaMemsetAsync(bad, 0, 4, st));
  long long blocks = (n + 1023) / 1024;
  if (blocks > 2 * num_sms()) blocks = 2 * num_sms();
  seg_count_kernel<<<(unsigned)blocks, 256, 0, st>>>(d_inter, n, n_user, off_u, bad);
  csr_scan_kernel<<<1, 1024, 0, st>>>(d_desc);
  int npass = 1;
  while (npass < 4 && (n_user - 1) >> (8 * npass)) ++npass;
  for (int pass = 0; pass < npass; ++pass) {            // grid.y = 1: shard 0, user side only
    radix_hist_kernel<<<dim3(kRadixBlocks, 1), kRadixThreads, 0, st>>>(d_desc, pass, npass, hist, nullptr);
    radix_scan_kernel<<<1, 256, 0, st>>>(hist, kRadixBlocks, nullptr);
    radix_scatter_kernel<<<dim3(kRadixBlocks, 1), kRadixThreads, 0, st>>>(d_desc, pass, npass, hist, nullptr);
  }
  seg_extract_kernel<<<(unsigned)blocks, 256, 0, st>>>(sorted, n, off_u, n_user, d_order, reinterpret_cast<long long*>(d_seg));
  URE_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------- per-user seen lists (recommendation)
// A user's training items in ascending order: the same stable radix sort, keyed first by item (the item side of the
// set-up's passes, one (shard, side) row per launch) and then by user, so that the user passes keep the item order.
namespace ure {
namespace {
__global__ void __launch_bounds__(kRadixThreads)
radix_hist_row_kernel(const ure_mf_shard_t* shards, int pass, int npass, int* __restrict__ hist, int y) {
  __shared__ int s_h[256];
  radix_hist_body(shards, pass, npass, hist, nullptr, s_h, blockIdx.x, y, gridDim.x);
}
__global__ void __launch_bounds__(256)
radix_scan_row_kernel(int* __restrict__ hist, int n_blocks, int y) {
  __shared__ int s_tot[256];
  radix_scan_body(hist, n_blocks, nullptr, s_tot, y);
}
__global__ void __launch_bounds__(kRadixThreads)
radix_scatter_row_kernel(const ure_mf_shard_t* shards, int pass, int npass, const int* __restrict__ hist, int y) {
  __shared__ int s_wh[kRadixWarps * 256];
  radix_scatter_body(shards, pass, npass, hist, nullptr, s_wh, blockIdx.x, y, gridDim.x);
}
__global__ void seen_extract_kernel(const ure_inter_t* __restrict__ sorted, long long n, const int32_t* __restrict__ off_u,
                                    int n_user, int32_t* __restrict__ items, long long* __restrict__ off) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) items[j] = sorted[j].item;
  for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u <= n_user; u += stride) off[u] = off_u[u];
}
}  // namespace
}  // namespace ure

extern "C" int64_t ure_seen_lists_scratch_bytes(int64_t n, int n_user) {
  using namespace ure;
  return 512 + seg_align(((int64_t)n_user + 2) * 4) + 3 * seg_align(n * 16) + seg_align(2 * 256ll * kRadixBlocks * 4) + 256;
}

extern "C" int ure_seen_lists(const ure_inter_t* d_inter, int64_t n, int n_user, int n_item, int64_t* d_off,
                              int32_t* d_items, void* d_scratch, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_off && d_scratch && n >= 0 && n_user > 0 && n_item > 0 && n < (1ll << 31) && (n == 0 || (d_inter && d_items)),
              URE_EINVAL, "ure_seen_lists: bad argument (n=%lld, n_user=%d, n_item=%d)", (long long)n, n_user, n_item);
  auto st = static_cast<cudaStream_t>(stream);
  char* base = static_cast<char*>(d_scratch);
  auto* d_desc = reinterpret_cast<ure_mf_shard_t*>(base);   // [0]: item passes, [1]: user passes
  auto* off_u = reinterpret_cast<int32_t*>(base + 512);
  char* p = base + 512 + seg_align(((int64_t)n_user + 2) * 4);
  auto* by_item = reinterpret_cast<ure_inter_t*>(p); p += seg_align(n * 16);
  auto* tmp = reinterpret_cast<ure_inter_t*>(p); p += seg_align(n * 16);
  auto* sorted = reinterpret_cast<ure_inter_t*>(p); p += seg_align(n * 16);
  auto* hist = reinterpret_cast<int*>(p); p += seg_align(2 * 256ll * kRadixBlocks * 4);
  int* bad = reinterpret_cast<int*>(p);
  ure_mf_shard_t h[2];
  memset(h, 0, sizeof(h));
  h[0].inter = d_inter; h[0].inter_i = by_item; h[0].tmp_i = tmp; h[0].n = (int32_t)n; h[0].n_item = n_item;
  h[1].inter = by_item; h[1].inter_u = sorted; h[1].tmp_u = tmp; h[1].off_u = off_u; h[1].n = (int32_t)n; h[1].n_user = n_user;
  URE_CUDA(cudaMemcpyAsync(d_desc, h, sizeof(h), cudaMemcpyHostToDevice, st));
  URE_CUDA(cudaMemsetAsync(off_u, 0, ((size_t)n_user + 2) * 4, st));
  URE_CUDA(cudaMemsetAsync(bad, 0, 4, st));
  long long blocks = (n + 1023) / 1024;
  if (blocks > 2 * num_sms()) blocks = 2 * num_sms();
  if (blocks < 1) blocks = 1;
  if (n > 0) {
    seg_count_kernel<<<(unsigned)blocks, 256, 0, st>>>(d_inter, n, n_user, off_u, bad);
    int npass = 1;
    while (npass < 4 && (n_item - 1) >> (8 * npass)) ++npass;
    for (int pass = 0; pass < npass; ++pass) {          // row y = 1: shard 0, item side
      radix_hist_row_kernel<<<kRadixBlocks, kRadixThreads, 0, st>>>(d_desc, pass, npass, hist, 1);
      radix_scan_row_kernel<<<1, 256, 0, st>>>(hist, kRadixBlocks, 1);
      radix_scatter_row_kernel<<<kRadixBlocks, kRadixThreads, 0, st>>>(d_desc, pass, npass, hist, 1);
    }
    npass = 1;
    while (npass < 4 && (n_user - 1) >> (8 * npass)) ++npass;
    for (int pass = 0; pass < npass; ++pass) {          // grid.y = 1: shard 0 of d_desc + 1, user side
      radix_hist_kernel<<<dim3(kRadixBlocks, 1), kRadixThreads, 0, st>>>(d_desc + 1, pass, npass, hist, nullptr);
      radix_scan_kernel<<<1, 256, 0, st>>>(hist, kRadixBlocks, nullptr);
      radix_scatter_kernel<<<dim3(kRadixBlocks, 1), kRadixThreads, 0, st>>>(d_desc + 1, pass, npass, hist, nullptr);
    }
  }
  csr_scan_kernel<<<1, 1024, 0, st>>>(d_desc + 1);
  seen_extract_kernel<<<(unsigned)blocks, 256, 0, st>>>(sorted, n, off_u, n_user, d_items, reinterpret_cast<long long*>(d_off));
  URE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int64_t ure_mf_owner_radix_bytes(int n_shards) { return 2ll * n_shards * 256 * ure::kRadixBlocks * 4; }

namespace ure {
int mf_owner_prepare_impl(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp, int epochs,
                          int max_rows, int32_t* d_radix_hist, void* d_workspace, void* stream, int flags);
}
extern "C" int ure_mf_owner_prepare(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp,
                                    int epochs, int max_rows, int32_t* d_radix_hist, void* d_workspace, void* stream) {
  return ure::mf_owner_prepare_impl(d_shards, n_shards, h_hp, epochs, max_rows, d_radix_hist, d_workspace, stream, 0);
}

// flags (the native batch runtime): 1 = the caller has just cleared the workspace; 2 = no plan kernel (the launch runs
// on remembered capacities, checked by the schedule pre-pass); 4 = no shard has explicit visiting orders; 8 = the whole
// set-up in one cooperative launch
int ure::mf_owner_prepare_impl(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp, int epochs,
                               int max_rows, int32_t* d_radix_hist, void* d_workspace, void* stream, int flags) {
  using namespace ure;
  URE_REQUIRE(d_shards && h_hp && d_workspace, URE_EINVAL, "ure_mf_owner_prepare: null argument");
  URE_REQUIRE(n_shards >= 1 && n_shards <= num_sms(), URE_EUNSUPPORTED,
              "ure_mf_owner_prepare: n_shards=%d outside [1,%d] (one CTA per shard at least)", n_shards, num_sms());
  auto st = static_cast<cudaStream_t>(stream);
  auto* ws = static_cast<OwnerWs*>(d_workspace);
  URE_REQUIRE(d_radix_hist && max_rows >= 1, URE_EINVAL, "ure_mf_owner_prepare: radix scratch / max_rows missing");
  const int blocks = 2 * num_sms();
  int npass = 1;
  while (npass < 4 && (max_rows - 1) >> (8 * npass)) ++npass;
  // max_rows bounds n_user and n_item of every shard: both tables' counters in shared memory when they fit 96 KB
  const int smem_rows = 2 * max_rows <= 24576 ? 2 * max_rows : 0;
  const int cb = smem_rows ? (num_sms() / n_shards > 0 ? num_sms() / n_shards : 1) : blocks;   // one wave of CTAs
  // flags & 8 (the batch runtime, small batches) or URE_SETUP_FUSED=1: one cooperative launch instead of 2 + 3 npass
  const char* const fe = getenv("URE_SETUP_FUSED");      // read per call: the tests compare both ways in one process
  const int fused_env = fe ? atoi(fe) : -1;
  bool fused = fused_env > 0 || (fused_env < 0 && (flags & 8));
  if (fused) {
    const int smem_ints = smem_rows > kRadixWarps * 256 ? smem_rows : kRadixWarps * 256;
    static int smem_set = 48 << 10;
    if (smem_ints * 4 > smem_set) {
      URE_CUDA(cudaFuncSetAttribute(owner_setup_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_ints * 4));
      smem_set = smem_ints * 4;
    }
    int occ = 0;
    URE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, owner_setup_kernel, kRadixThreads, (size_t)smem_ints * 4));
    if (occ < 1) fused = false;
    else {
      if (!(flags & 1)) URE_CUDA(cudaMemsetAsync(ws->unsorted, 0, sizeof(ws->unsorted), st));
      const int per_sm = occ < 4 ? occ : 4;
      int n_sh = n_shards, sr = smem_rows, cbv = cb, np = npass;
      const ure_mf_shard_t* dsh = d_shards;
      int32_t* hist = d_radix_hist;
      unsigned* uns = ws->unsorted;
      void* args[] = {&dsh, &n_sh, &sr, &cbv, &np, &hist, &uns};
      URE_CUDA(cudaLaunchCooperativeKernel((void*)owner_setup_kernel, dim3(per_sm * num_sms()), dim3(kRadixThreads), args,
                                           (size_t)smem_ints * 4, st));
    }
  }
  if (!fused) {
    if (smem_rows)
      URE_CUDA(cudaFuncSetAttribute(csr_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_rows * 4));
    if (!(flags & 1)) URE_CUDA(cudaMemsetAsync(ws->unsorted, 0, sizeof(ws->unsorted), st));
    csr_count_kernel<<<dim3(cb, n_shards), 1024, (size_t)smem_rows * 4, st>>>(d_shards, smem_rows, ws->unsorted);
    csr_scan_kernel<<<2 * n_shards, 1024, 0, st>>>(d_shards);
    for (int pass = 0; pass < npass; ++pass) {
      radix_hist_kernel<<<dim3(kRadixBlocks, 2 * n_shards), kRadixThreads, 0, st>>>(d_shards, pass, npass, d_radix_hist, ws->unsorted);
      radix_scan_kernel<<<2 * n_shards, 256, 0, st>>>(d_radix_hist, kRadixBlocks, ws->unsorted);
      radix_scatter_kernel<<<dim3(kRadixBlocks, 2 * n_shards), kRadixThreads, 0, st>>>(d_shards, pass, npass, d_radix_hist, ws->unsorted);
    }
  }
  if (!(flags & 4)) perm_inverse_kernel<<<dim3(blocks, n_shards), 256, 0, st>>>(d_shards, epochs);
  int avail = 0;
  if (int rc = max_dyn_smem(&avail)) return rc;
  if (!(flags & 1)) {                      // a workspace of unknown content: reset the plan fields
    const int head[6] = {0, 0, 0, 0, 0, 0};
    URE_CUDA(cudaMemcpyAsync(ws, head, sizeof(head), cudaMemcpyHostToDevice, st));
  }
  if (!(flags & 2)) plan_kernel<<<num_sms(), 32, 0, st>>>(d_shards, n_shards, h_hp->batch, avail, ws);
  URE_CUDA(cudaGetLastError());
  return 0;
}
