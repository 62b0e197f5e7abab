// RUNS schedule of the fused MF training step (ure_mf_hparams_t::mode == URE_MF_RUNS): owner-computes for tables
// that do not fit shared memory (BASELINE config C4: 10 M users x 1 M items, d = 128, 8 shards per GPU).
//
// Same arithmetic as the other schedules (baseTrain, reference method/utils.py:58-98, + the dense
// optim.SGD(momentum, weight_decay) of scratch.py:65-68 -- a row that receives no gradient still decays every
// step; as in the LAZY schedule it catches up in closed form, [w;buf] <- M^n [w;buf], when it is next used).
// What changes is the data movement.  LAZY scatters gradients with L2 atomics into dense gradient arrays and then
// re-reads weights, momentum and gradients of every touched row: ~10 KB of DRAM traffic per interaction at d = 128
// (ncu: 97 GB per 9.6 M interactions) against 2 KB algorithmic.  Here:
//   * the shard's records exist sorted by user and sorted by item (ure_mf_owner_prepare); per epoch a stable
//     counting sort by step (ure_mf_runs_schedule) leaves, for every step, the batch's interactions as two lists in
//     row order -- consecutive entries with the same row form a RUN;
//   * a warp owns whole runs: it reads its row once (weights + momentum, advanced to the current step in
//     registers), gathers the OTHER table's row for every entry of the run (also advanced), sums the gradient in
//     registers and writes the updated row once.  No atomics, no gradient arrays, no touched lists.  Every
//     interaction is processed twice (user side and item side), as in the OWNER schedule;
//   * batch-synchronous semantics with ONE grid barrier per step: a row has two slots and a 64-bit tag
//     {steps applied to the previous version, steps applied to the current version, current slot}.  The writer of
//     step t reads slot `cur`, writes slot `cur ^ 1` and then the tag; a reader of step t that sees a tag saying
//     "t + 1 steps applied" knows the row was rewritten during this very step and takes the previous version --
//     the slot the writer did not touch.  Either way it reads the pre-step weights.
//   Traffic per interaction: 2 x (1 KB row + tag) gathers + ~1.7 touched rows x 2 KB  ~ 5.4 KB at d = 128.
#include "common.cuh"
#include "feistel.cuh"

namespace ure {
namespace {

constexpr int kRunThreads = 512;           // 16 warps, no spills (~120 registers: two entries of a run in flight per warp)
constexpr int KM = URE_MAX_SHARDS;
constexpr int kRunTile = 32768;          // slots per CTA of the schedule pre-pass
constexpr int kRunSortThreads = 512;
constexpr int kRunSortWarps = kRunSortThreads / 32;
constexpr int kRunMaxBins = 1024;        // steps per epoch the one-pass counting sort handles

struct RunsWs {
  unsigned barrier;
  unsigned pad[63];
};

__device__ __forceinline__ float4 adv_w(const float4 c, const float4 w, const float4 b) {
  return make_float4(fmaf(c.x, w.x, c.y * b.x), fmaf(c.x, w.y, c.y * b.y), fmaf(c.x, w.z, c.y * b.z),
                     fmaf(c.x, w.w, c.y * b.w));
}
__device__ __forceinline__ float4 adv_b(const float4 c, const float4 w, const float4 b) {
  return make_float4(fmaf(c.z, w.x, c.w * b.x), fmaf(c.z, w.y, c.w * b.y), fmaf(c.z, w.z, c.w * b.z),
                     fmaf(c.z, w.w, c.w * b.w));
}

// tag = (steps applied to the previous version) << 32 | (steps applied to the current version) << 1 | current slot
__device__ __forceinline__ void pick_version(unsigned long long tag, int t, int& slot, int& last) {
  const unsigned cur = (unsigned)tag;
  slot = (int)(cur & 1u);
  last = (int)(cur >> 1);
  if (last == t + 1) {                    // rewritten during this step: the previous version is the pre-step one
    slot ^= 1;
    last = (int)(tag >> 32);
  }
}

// ---------------------------------------------------------------- schedule pre-pass: stable counting sort by step
// job = (shard, side, window row).  Grid (tiles, jobs).
struct RunJob {
  const ure_inter_t* rec;   // inter_u or inter_i
  uint32_t* list;           // [n] output: slots grouped by step
  int32_t* loff;            // [spe_cap + 1] output: first entry of every step (loff[spe] = n)
  unsigned short* steps;    // [n] scratch: step of every slot
  int n, spe, epoch, shard;
};

__device__ __forceinline__ bool run_job(const ure_mf_shard_t* shards, const ure_mf_hparams_t& hp, int epochs,
                                        long long step0, unsigned short* steps_all, long long steps_stride, RunJob& j) {
  const int job = blockIdx.y;
  const int rows = hp.runs_rows;
  const int s = job / (2 * rows), rest = job % (2 * rows), side = rest / rows, r = rest % rows;
  const ure_mf_shard_t& sh = shards[s];
  const ure_mf_runs_t& rs = hp.runs[s];
  j.n = sh.n;
  j.spe = (sh.n + hp.batch - 1) / hp.batch;
  j.shard = s;
  if (j.spe == 0) return false;
  j.epoch = (int)(step0 / j.spe) + r;
  if (j.epoch >= epochs) return false;
  j.rec = side ? sh.inter_i : sh.inter_u;
  j.list = (side ? rs.list_i : rs.list_u) + (long long)r * sh.n;
  j.loff = (side ? rs.loff_i : rs.loff_u) + (long long)r * (hp.runs_spe_cap + 1);
  j.steps = steps_all + (long long)job * steps_stride;
  return true;
}

// hist [jobs][tiles][bins]
__global__ void __launch_bounds__(kRunSortThreads)
runs_hist_kernel(const ure_mf_shard_t* __restrict__ shards, ure_mf_hparams_t hp, int epochs, long long step0,
                 unsigned short* __restrict__ steps_all, long long steps_stride, int bins, int* __restrict__ hist) {
  extern __shared__ int s_h[];
  RunJob j;
  if (!run_job(shards, hp, epochs, step0, steps_all, steps_stride, j)) return;
  const long long t0 = (long long)blockIdx.x * kRunTile;
  if (t0 >= j.n) return;
  const long long t1 = min((long long)j.n, t0 + kRunTile);
  for (int x = threadIdx.x; x < bins; x += blockDim.x) s_h[x] = 0;
  __syncthreads();
  const ure_mf_shard_t& sh = shards[j.shard];
  FeistelDomain dom;
  dom.init((uint32_t)j.n);
  FeistelKeys ks;
  ks.init(perm_key(sh.perm_seed, (uint32_t)sh.shard_id, (uint32_t)j.epoch));
  const int32_t* pinv = sh.perm_inv ? sh.perm_inv + (long long)j.epoch * j.n : nullptr;
  const uint32_t B = (uint32_t)hp.batch;
  constexpr int NI = 4;
  for (long long base = t0 + threadIdx.x; base < t1; base += (long long)NI * blockDim.x) {
    uint32_t x[NI];
    bool live[NI];
#pragma unroll
    for (int u = 0; u < NI; ++u) {
      const long long sl = base + (long long)u * blockDim.x;
      live[u] = sl < t1;
      x[u] = live[u] ? (uint32_t)__ldg(&j.rec[sl].pad) : 0u;
    }
    if (pinv) {
#pragma unroll
      for (int u = 0; u < NI; ++u)
        if (live[u]) x[u] = (uint32_t)__ldg(pinv + x[u]);
    } else {
      feistel_inverse_n<NI>(dom, ks, x, live);
    }
#pragma unroll
    for (int u = 0; u < NI; ++u) {
      if (!live[u]) continue;
      const uint32_t q = x[u] / B;
      j.steps[base + (long long)u * blockDim.x] = (unsigned short)q;
      atomicAdd(&s_h[q], 1);
    }
  }
  __syncthreads();
  int* out = hist + ((long long)blockIdx.y * gridDim.x + blockIdx.x) * bins;
  for (int x = threadIdx.x; x < bins; x += blockDim.x) out[x] = s_h[x];
}

// per job: exclusive scan of hist in (step, tile) order, in place; thread = step
__global__ void __launch_bounds__(kRunMaxBins)
runs_scan_kernel(const ure_mf_shard_t* __restrict__ shards, ure_mf_hparams_t hp, int epochs, long long step0, int tiles,
                 int bins, int* __restrict__ hist) {
  __shared__ int s_tot[kRunMaxBins];
  __shared__ int s_warp[32];
  RunJob j;
  if (!run_job(shards, hp, epochs, step0, nullptr, 0, j)) return;
  const int used = (j.n + kRunTile - 1) / kRunTile;      // tiles of this job that ran
  const int b = threadIdx.x;
  int* h = hist + (long long)blockIdx.y * tiles * bins + b;
  int tot = 0;
  if (b < bins)
    for (int t = 0; t < used; ++t) tot += h[(long long)t * bins];
  // block exclusive scan over the steps
  const int lane = b & 31, warp = b >> 5;
  int inc = tot;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int a = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += a;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = s_warp[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int a = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += a;
    }
    s_warp[lane] = w;
  }
  __syncthreads();
  int run = inc - tot + (warp > 0 ? s_warp[warp - 1] : 0);
  if (b <= j.spe) j.loff[b] = b < j.spe ? run : j.n;
  if (b < bins)
    for (int t = 0; t < used; ++t) {
      const int v = h[(long long)t * bins];
      h[(long long)t * bins] = run;
      run += v;
    }
  (void)s_tot;
}

// stable scatter of the CTA's tile: every warp owns a contiguous range; per-warp step counts -> per-warp cursors
__global__ void __launch_bounds__(kRunSortThreads)
runs_scatter_kernel(const ure_mf_shard_t* __restrict__ shards, ure_mf_hparams_t hp, int epochs, long long step0,
                    unsigned short* __restrict__ steps_all, long long steps_stride, int bins, const int* __restrict__ hist) {
  extern __shared__ int s_wh[];            // [warps][bins]
  RunJob j;
  if (!run_job(shards, hp, epochs, step0, steps_all, steps_stride, j)) return;
  const long long t0 = (long long)blockIdx.x * kRunTile;
  if (t0 >= j.n) return;
  const long long t1 = min((long long)j.n, t0 + kRunTile);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned lt = (1u << lane) - 1u;
  for (int x = threadIdx.x; x < kRunSortWarps * bins; x += blockDim.x) s_wh[x] = 0;
  __syncthreads();
  const long long per = ((t1 - t0) + kRunSortWarps - 1) / kRunSortWarps;
  const long long w0 = min(t1, t0 + per * warp), w1 = min(t1, w0 + per);
  int* mine = s_wh + warp * bins;
  for (long long s0 = w0; s0 < w1; s0 += 32) {
    const long long sl = s0 + lane;
    const bool in = sl < w1;
    const int q = in ? (int)j.steps[sl] : 0;
    const unsigned act = __ballot_sync(0xffffffffu, in);
    if (in) {
      const unsigned same = __match_any_sync(act, q);
      if (lane == __ffs(same) - 1) mine[q] += __popc(same);
    }
    __syncwarp();
  }
  __syncthreads();
  const int* base = hist + ((long long)blockIdx.y * gridDim.x + blockIdx.x) * bins;
  for (int q = threadIdx.x; q < bins; q += blockDim.x) {
    int run = base[q];
    for (int w = 0; w < kRunSortWarps; ++w) {
      const int t = s_wh[w * bins + q];
      s_wh[w * bins + q] = run;
      run += t;
    }
  }
  __syncthreads();
  for (long long s0 = w0; s0 < w1; s0 += 32) {
    const long long sl = s0 + lane;
    const bool in = sl < w1;
    const int q = in ? (int)j.steps[sl] : 0;
    const unsigned act = __ballot_sync(0xffffffffu, in);
    if (in) {
      const unsigned same = __match_any_sync(act, q);
      j.list[mine[q] + __popc(same & lt)] = (uint32_t)sl;
      __syncwarp(act);
      if (lane == __ffs(same) - 1) mine[q] += __popc(same);
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------- row slots <-> the public tables
// init: slot 0 of every row <- [P row | bufP row], tag 0 (no step applied, current slot 0)
template <int D>
__global__ void runs_init_kernel(const ure_mf_shard_t* __restrict__ shards, const ure_mf_runs_t* __restrict__ runs) {
  const ure_mf_shard_t& sh = shards[blockIdx.y];
  const ure_mf_runs_t& rs = runs[blockIdx.y];
  constexpr int CH = D / 4;
  const long long rows = (long long)sh.n_user + sh.n_item;
  for (long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x; x < rows * CH; x += (long long)gridDim.x * blockDim.x) {
    const long long r = x / CH;
    const int c = (int)(x % CH);
    const bool it = r >= sh.n_user;
    const long long row = it ? r - sh.n_user : r;
    const float* W = it ? sh.Q : sh.P;
    const float* Bf = it ? sh.bufQ : sh.bufP;
    float* S = it ? rs.slotQ : rs.slotP;
    const float4 w = __ldg(reinterpret_cast<const float4*>(W + row * D) + c);
    const float4 b = __ldg(reinterpret_cast<const float4*>(Bf + row * D) + c);
    *(reinterpret_cast<float4*>(S + row * 2 * D) + c) = w;
    *(reinterpret_cast<float4*>(S + row * 2 * D + D) + c) = b;
    if (c == 0) (it ? rs.metaQ : rs.metaP)[row] = 0ull;
  }
}

// flush: every row advanced to `done_s` steps, written to the public tables (the slots stay the source of truth)
template <int D>
__global__ void runs_flush_kernel(const ure_mf_shard_t* __restrict__ shards, const ure_mf_runs_t* __restrict__ runs,
                                  ure_mf_hparams_t hp, int epochs, long long step_now) {
  const ure_mf_shard_t& sh = shards[blockIdx.y];
  const ure_mf_runs_t& rs = runs[blockIdx.y];
  constexpr int CH = D / 4;
  const long long spe = (sh.n + hp.batch - 1) / hp.batch;
  const int done = (int)(spe * epochs < step_now ? spe * epochs : step_now);
  const float4* decay = reinterpret_cast<const float4*>(hp.decay);
  const long long rows = (long long)sh.n_user + sh.n_item;
  for (long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x; x < rows * CH; x += (long long)gridDim.x * blockDim.x) {
    const long long r = x / CH;
    const int c = (int)(x % CH);
    const bool it = r >= sh.n_user;
    const long long row = it ? r - sh.n_user : r;
    const long long n_rows = it ? sh.n_item : sh.n_user;
    const unsigned long long tag = (it ? rs.metaQ : rs.metaP)[row];
    const int slot = (int)(tag & 1ull), last = (int)((unsigned)tag >> 1);
    const float* S = (it ? rs.slotQ : rs.slotP) + ((long long)slot * n_rows + row) * 2 * D;
    const float4 w = *(reinterpret_cast<const float4*>(S) + c);
    const float4 b = *(reinterpret_cast<const float4*>(S + D) + c);
    const float4 cf = __ldg(decay + max(0, done - last));
    *(reinterpret_cast<float4*>((it ? sh.Q : sh.P) + row * D) + c) = adv_w(cf, w, b);
    *(reinterpret_cast<float4*>((it ? sh.bufQ : sh.bufP) + row * D) + c) = adv_b(cf, w, b);
  }
}

// ---------------------------------------------------------------- the training kernel
template <typename T>
__device__ __forceinline__ int find_seg(const T* prefix, int nseg, T x) {
  int lo = 0, hi = nseg;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (prefix[mid] <= x) lo = mid; else hi = mid;
  }
  return lo;
}

template <int D>
__global__ void __launch_bounds__(kRunThreads, 1)
mf_runs_kernel(const ure_mf_shard_t* __restrict__ shards, int K, ure_mf_hparams_t hp, int epochs, long long step_begin,
               long long step_end, RunsWs* ws) {
  constexpr int G = D / 4;                 // lanes that carry a row (16-byte chunk each)
  constexpr unsigned FULL = 0xffffffffu;
  __shared__ int s_unit_prefix[2 * KM + 1];
  __shared__ int s_seg0[2 * KM], s_seg1[2 * KM], s_epoch[KM];
  __shared__ float s_sse_acc[KM];
  const int tid = threadIdx.x, lane = tid & 31;
  const bool act = lane < G;
  const float4* __restrict__ decay = reinterpret_cast<const float4*>(hp.decay);
  const float wd = hp.weight_decay, mu = hp.momentum, nlr = -hp.lr0;
  const int n_warps = (int)(((long long)gridDim.x * kRunThreads) >> 5);
  const int gwarp = (tid >> 5) * (int)gridDim.x + (int)blockIdx.x;      // CTA-minor: few units still use every SM
  unsigned bar_target = 0;
  for (int s = tid; s < K; s += kRunThreads) s_sse_acc[s] = 0.f;

  for (long long t = step_begin; t < step_end; ++t) {
    const int tt = (int)t;
    // ---- step tables: the two list segments of every shard and their prefix in units of 32 entries
    if (tid < 32) {
      int carry = 0;
      for (int base = 0; base < 2 * K; base += 32) {
        const int seg = base + lane;
        int units = 0;
        if (seg < 2 * K) {
          const int s = seg >> 1, side = seg & 1;
          const ure_mf_shard_t& sh = shards[s];
          const int spe = (sh.n + hp.batch - 1) / hp.batch;
          int a = 0, b = 0, ep = -1;
          if (spe > 0 && t < (long long)spe * epochs) {
            ep = (int)(t / spe);
            const int k = (int)(t % spe), row = ep - (int)(hp.runs_step0 / spe);
            if (row >= 0 && row < hp.runs_rows) {
              const int32_t* lo = (side ? hp.runs[s].loff_i : hp.runs[s].loff_u) + (long long)row * (hp.runs_spe_cap + 1);
              a = __ldg(lo + k) + row * sh.n;           // positions inside the window's list array
              b = __ldg(lo + k + 1) + row * sh.n;
            } else {
              ep = -2;                                   // outside the scheduled window: the host made a mistake
            }
          }
          s_seg0[seg] = a; s_seg1[seg] = b;
          if (side == 0) s_epoch[s] = ep;
          units = (b - a + 31) >> 5;
        }
        int v = units;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int x = __shfl_up_sync(FULL, v, o); if (lane >= o) v += x; }
        if (seg < 2 * K) s_unit_prefix[seg + 1] = v + carry;
        carry += __shfl_sync(FULL, v, 31);
      }
      if (lane == 0) s_unit_prefix[0] = 0;
    }
    __syncthreads();
    const int total_units = s_unit_prefix[2 * K];

    for (int unit = gwarp; unit < total_units; unit += n_warps) {
      const int seg = find_seg(s_unit_prefix, 2 * K, unit);
      const int s = seg >> 1, side = seg & 1;
      const ure_mf_shard_t& sh = shards[s];
      const ure_mf_runs_t& rs = hp.runs[s];
      const int seg0 = s_seg0[seg], seg1 = s_seg1[seg];
      const int e0 = seg0 + ((unit - s_unit_prefix[seg]) << 5);
      const uint32_t* __restrict__ list = side ? rs.list_i : rs.list_u;
      const ure_inter_t* __restrict__ rec = side ? sh.inter_i : sh.inter_u;
      float* const S_own = side ? rs.slotQ : rs.slotP;
      const float* const S_oth = side ? rs.slotP : rs.slotQ;
      unsigned long long* const T_own = side ? rs.metaQ : rs.metaP;
      const unsigned long long* const T_oth = side ? rs.metaP : rs.metaQ;
      const long long rows_own = side ? sh.n_item : sh.n_user, rows_oth = side ? sh.n_user : sh.n_item;

      // the run in progress
      int cur_row = -1, cur_slot = 0, cur_last = 0;
      float4 w_own = make_float4(0.f, 0.f, 0.f, 0.f), b_own = w_own, g = w_own;
      float sse_l = 0.f;
      auto finalize = [&]() {
        if (cur_row < 0) return;
        // torch SGD: d_p = g + wd*w (fma); buf = buf*mu + d_p; w = w + (-lr)*buf (fma)
        g.x = fmaf(wd, w_own.x, g.x); g.y = fmaf(wd, w_own.y, g.y); g.z = fmaf(wd, w_own.z, g.z); g.w = fmaf(wd, w_own.w, g.w);
        b_own.x = __fadd_rn(__fmul_rn(b_own.x, mu), g.x); b_own.y = __fadd_rn(__fmul_rn(b_own.y, mu), g.y);
        b_own.z = __fadd_rn(__fmul_rn(b_own.z, mu), g.z); b_own.w = __fadd_rn(__fmul_rn(b_own.w, mu), g.w);
        w_own.x = fmaf(nlr, b_own.x, w_own.x); w_own.y = fmaf(nlr, b_own.y, w_own.y);
        w_own.z = fmaf(nlr, b_own.z, w_own.z); w_own.w = fmaf(nlr, b_own.w, w_own.w);
        float* dst = S_own + ((long long)(cur_slot ^ 1) * rows_own + cur_row) * 2 * D;
        if (act) {
          __stcg(reinterpret_cast<float4*>(dst) + lane, w_own);
          __stcg(reinterpret_cast<float4*>(dst + D) + lane, b_own);
        }
        __syncwarp();
        if (lane == 0) {
          const unsigned long long tag = ((unsigned long long)(unsigned)cur_last << 32) |
                                         (unsigned long long)(((unsigned)(tt + 1) << 1) | (unsigned)(cur_slot ^ 1));
          __stcg(T_own + cur_row, tag);
        }
        cur_row = -1;
      };

      int carry_own = -2;                 // own row of the entry before the chunk
      if (e0 > seg0) {
        const uint32_t sp = __ldg(list + e0 - 1);
        const int4 rp = ld_stream_i4(rec + sp);
        carry_own = side ? rp.y : rp.x;
      }
      for (int base = e0;; base += 32) {
        const int e = base + lane;
        const bool valid = e < seg1;
        int own = -1, oth = 0;
        float rating = 0.f;
        unsigned long long tag_o = 0ull, tag_m = 0ull;
        if (valid) {
          const int4 r4 = ld_stream_i4(rec + __ldg(list + e));
          own = side ? r4.y : r4.x;
          oth = side ? r4.x : r4.y;
          rating = __int_as_float(r4.z);
          tag_o = __ldcg(T_oth + oth);
        }
        int prev = __shfl_up_sync(FULL, own, 1);
        if (lane == 0) prev = carry_own;
        const bool is_start = valid && own != prev;
        if (is_start) tag_m = __ldcg(T_own + own);
        const unsigned start_mask = __ballot_sync(FULL, is_start);
        const unsigned valid_mask = __ballot_sync(FULL, valid);
        unsigned proc;
        bool more;                         // the run goes on into the next chunk
        if (base == e0) {
          // the unit itself: everything from its first run start on (the entries before belong to a run of the
          // previous unit's warp)
          proc = start_mask ? (valid_mask & ~((1u << (__ffs(start_mask) - 1)) - 1u)) : 0u;
          more = proc != 0u && valid_mask == FULL;
        } else {
          // continuation: only the tail of the run in progress
          const unsigned stop = start_mask | ~valid_mask;
          proc = stop ? ((1u << (__ffs(stop) - 1)) - 1u) : FULL;
          more = stop == 0u;
        }
        carry_own = __shfl_sync(FULL, own, 31);

        // entries of `proc` in order, the next one's rows in flight while the current one is consumed
        struct Ent { float4 ow, ob, mw, mb; };
        auto issue = [&](int jx, Ent& E, int& o_last, int& m_slot, int& m_last) {
          const int oth_j = __shfl_sync(FULL, oth, jx), own_j = __shfl_sync(FULL, own, jx);
          const unsigned long long to = __shfl_sync(FULL, tag_o, jx), tm = __shfl_sync(FULL, tag_m, jx);
          int o_slot;
          pick_version(to, tt, o_slot, o_last);
          const float* src = S_oth + ((long long)o_slot * rows_oth + oth_j) * 2 * D;
          E.ow = make_float4(0.f, 0.f, 0.f, 0.f); E.ob = E.ow; E.mw = E.ow; E.mb = E.ow;
          if (act) {
            E.ow = __ldcg(reinterpret_cast<const float4*>(src) + lane);
            E.ob = __ldcg(reinterpret_cast<const float4*>(src + D) + lane);
          }
          m_slot = (int)(tm & 1ull);
          m_last = (int)((unsigned)tm >> 1);
          if ((start_mask >> jx) & 1u) {
            const float* ms = S_own + ((long long)m_slot * rows_own + own_j) * 2 * D;
            if (act) {
              E.mw = __ldcg(reinterpret_cast<const float4*>(ms) + lane);
              E.mb = __ldcg(reinterpret_cast<const float4*>(ms + D) + lane);
            }
          }
        };
        auto consume = [&](int jx, const Ent& E, int o_last, int m_slot, int m_last) {
          if ((start_mask >> jx) & 1u) {
            finalize();
            cur_row = __shfl_sync(FULL, own, jx);
            cur_slot = m_slot;
            cur_last = m_last;
            const float4 cf = __ldg(decay + (tt - m_last));
            w_own = adv_w(cf, E.mw, E.mb);
            b_own = adv_b(cf, E.mw, E.mb);
            g = make_float4(0.f, 0.f, 0.f, 0.f);
          }
          const float4 wo = adv_w(__ldg(decay + (tt - o_last)), E.ow, E.ob);
          float dot = w_own.x * wo.x;
          dot = fmaf(w_own.y, wo.y, dot);
          dot = fmaf(w_own.z, wo.z, dot);
          dot = fmaf(w_own.w, wo.w, dot);
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(FULL, dot, o);
          const float err = dot - __shfl_sync(FULL, rating, jx);
          const float ge = 2.f * err;
          g.x = fmaf(ge, wo.x, g.x); g.y = fmaf(ge, wo.y, g.y); g.z = fmaf(ge, wo.z, g.z); g.w = fmaf(ge, wo.w, g.w);
          if (side == 0) sse_l = fmaf(err, err, sse_l);
        };
        if (base != e0 && cur_row < 0) proc = 0u;           // nothing in progress: nothing to continue
        unsigned m = proc;
        Ent A, Bq;
        int a_ol = 0, a_ms = 0, a_ml = 0, b_ol = 0, b_ms = 0, b_ml = 0, ja = -1, jb = -1;
        if (m) { ja = __ffs(m) - 1; m &= m - 1; issue(ja, A, a_ol, a_ms, a_ml); }
        while (ja >= 0) {
          if (m) { jb = __ffs(m) - 1; m &= m - 1; issue(jb, Bq, b_ol, b_ms, b_ml); } else jb = -1;
          consume(ja, A, a_ol, a_ms, a_ml);
          if (jb < 0) break;
          if (m) { ja = __ffs(m) - 1; m &= m - 1; issue(ja, A, a_ol, a_ms, a_ml); } else ja = -1;
          consume(jb, Bq, b_ol, b_ms, b_ml);
        }
        if (!more || cur_row < 0) break;
      }
      finalize();
      if (side == 0 && lane == 0 && sse_l != 0.f) atomicAdd(&s_sse_acc[s], sse_l);
    }
    __syncthreads();
    for (int s = tid; s < K; s += kRunThreads) {
      const float v = s_sse_acc[s];
      if (v != 0.f && s_epoch[s] >= 0) atomicAdd(shards[s].sse + s_epoch[s], (double)v);
      s_sse_acc[s] = 0.f;
    }
    grid_barrier(&ws->barrier, bar_target);
  }
}

template <int D>
int launch_runs(const ure_mf_shard_t* d_shards, int K, const ure_mf_hparams_t& hp, int epochs, long long s0, long long s1,
                RunsWs* ws, cudaStream_t st) {
  void* kern = (void*)mf_runs_kernel<D>;
  int occ = 0;
  URE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kRunThreads, 0));
  URE_REQUIRE(occ >= 1, URE_ECOOP, "mf_runs_kernel<%d> cannot be resident", D);
  URE_CUDA(cudaMemsetAsync(&ws->barrier, 0, sizeof(unsigned), st));
  void* args[] = {(void*)&d_shards, (void*)&K, (void*)&hp, (void*)&epochs, (void*)&s0, (void*)&s1, (void*)&ws};
  URE_CUDA(cudaLaunchCooperativeKernel(kern, dim3(num_sms()), dim3(kRunThreads), args, 0, st));
  return 0;
}

int check_runs(const ure_mf_hparams_t* hp, int epochs, const char* who) {
  URE_REQUIRE(hp && hp->runs && hp->runs_rows >= 1 && hp->runs_spe_cap >= 1, URE_EINVAL,
              "%s: hparams.runs / runs_rows / runs_spe_cap missing", who);
  URE_REQUIRE(hp->runs_spe_cap < kRunMaxBins, URE_EUNSUPPORTED, "%s: %d steps per epoch (at most %d)", who,
              hp->runs_spe_cap, kRunMaxBins - 1);
  URE_REQUIRE(hp->decay && hp->decay_len > 0, URE_EINVAL, "%s: the decay table (M^n) is missing", who);
  URE_REQUIRE(epochs <= hp->lr_step, URE_EUNSUPPORTED,
              "%s: the learning rate must be constant over the training (epochs <= lr_step)", who);
  URE_REQUIRE(hp->d == 8 || hp->d == 16 || hp->d == 32 || hp->d == 64 || hp->d == 128, URE_EUNSUPPORTED,
              "%s: d=%d not in {8,16,32,64,128}", who, hp->d);
  return 0;
}

}  // namespace

// called by ure_mf_train when hparams.mode == URE_MF_RUNS
int mf_train_runs(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* hp, int epochs,
                  long long step_begin, long long step_end, void* d_workspace, cudaStream_t st) {
  if (int rc = check_runs(hp, epochs, "ure_mf_train(runs)")) return rc;
  URE_REQUIRE(hp->decay_len > step_end, URE_EINVAL, "ure_mf_train(runs): decay table must cover %lld steps (has %d)",
              (long long)step_end, hp->decay_len);
  URE_REQUIRE(hp->runs_step0 <= step_begin, URE_EINVAL, "ure_mf_train(runs): no schedule for step %lld", step_begin);
  if (step_end <= step_begin) return 0;
  auto* ws = static_cast<RunsWs*>(d_workspace);
  switch (hp->d) {
    case 8: return launch_runs<8>(d_shards, n_shards, *hp, epochs, step_begin, step_end, ws, st);
    case 16: return launch_runs<16>(d_shards, n_shards, *hp, epochs, step_begin, step_end, ws, st);
    case 32: return launch_runs<32>(d_shards, n_shards, *hp, epochs, step_begin, step_end, ws, st);
    case 64: return launch_runs<64>(d_shards, n_shards, *hp, epochs, step_begin, step_end, ws, st);
    default: return launch_runs<128>(d_shards, n_shards, *hp, epochs, step_begin, step_end, ws, st);
  }
}

}  // namespace ure

extern "C" int64_t ure_mf_runs_scratch_bytes(int n_shards, int64_t max_n, int rows, int spe_cap) {
  const int64_t tiles = (max_n + ure::kRunTile - 1) / ure::kRunTile;
  const int64_t jobs = 2ll * n_shards * rows;
  return jobs * ((max_n + 7) / 8 * 8) * 2 + jobs * (tiles > 0 ? tiles : 1) * (spe_cap + 1) * 4 + 256;
}

extern "C" int ure_mf_runs_init(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_shards && h_hp && h_hp->runs, URE_EINVAL, "ure_mf_runs_init: null argument");
  auto st = static_cast<cudaStream_t>(stream);
  const dim3 grid(num_sms() * 4, n_shards);
  switch (h_hp->d) {
    case 8: runs_init_kernel<8><<<grid, 256, 0, st>>>(d_shards, h_hp->runs); break;
    case 16: runs_init_kernel<16><<<grid, 256, 0, st>>>(d_shards, h_hp->runs); break;
    case 32: runs_init_kernel<32><<<grid, 256, 0, st>>>(d_shards, h_hp->runs); break;
    case 64: runs_init_kernel<64><<<grid, 256, 0, st>>>(d_shards, h_hp->runs); break;
    case 128: runs_init_kernel<128><<<grid, 256, 0, st>>>(d_shards, h_hp->runs); break;
    default: set_error("ure_mf_runs_init: d=%d not in {8,16,32,64,128}", h_hp->d); return URE_EUNSUPPORTED;
  }
  URE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int ure_mf_runs_schedule(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp, int epochs,
                                    int64_t step0, int64_t max_n, void* d_scratch, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_shards && d_scratch && max_n >= 0, URE_EINVAL, "ure_mf_runs_schedule: null argument");
  if (int rc = check_runs(h_hp, epochs, "ure_mf_runs_schedule")) return rc;
  if (max_n == 0) return 0;
  auto st = static_cast<cudaStream_t>(stream);
  const int bins = h_hp->runs_spe_cap + 1;
  const int tiles = (int)((max_n + kRunTile - 1) / kRunTile);
  const int jobs = 2 * n_shards * h_hp->runs_rows;
  const long long stride = (max_n + 7) / 8 * 8;
  auto* steps = static_cast<unsigned short*>(d_scratch);
  int* hist = reinterpret_cast<int*>(static_cast<char*>(d_scratch) + (size_t)jobs * stride * 2);
  ure_mf_hparams_t hp = *h_hp;
  hp.runs_step0 = step0;
  URE_CUDA(cudaFuncSetAttribute(runs_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kRunSortWarps * bins * 4));
  runs_hist_kernel<<<dim3(tiles, jobs), kRunSortThreads, (size_t)bins * 4, st>>>(d_shards, hp, epochs, step0, steps, stride, bins, hist);
  runs_scan_kernel<<<dim3(1, jobs), kRunMaxBins, 0, st>>>(d_shards, hp, epochs, step0, tiles, bins, hist);
  runs_scatter_kernel<<<dim3(tiles, jobs), kRunSortThreads, (size_t)kRunSortWarps * bins * 4, st>>>(d_shards, hp, epochs, step0,
                                                                                              steps, stride, bins, hist);
  URE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int ure_mf_runs_flush(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp, int epochs,
                                 int64_t step_now, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_shards, URE_EINVAL, "ure_mf_runs_flush: null argument");
  if (int rc = check_runs(h_hp, epochs, "ure_mf_runs_flush")) return rc;
  auto st = static_cast<cudaStream_t>(stream);
  const dim3 grid(num_sms() * 4, n_shards);
  switch (h_hp->d) {
    case 8: runs_flush_kernel<8><<<grid, 256, 0, st>>>(d_shards, h_hp->runs, *h_hp, epochs, step_now); break;
    case 16: runs_flush_kernel<16><<<grid, 256, 0, st>>>(d_shards, h_hp->runs, *h_hp, epochs, step_now); break;
    case 32: runs_flush_kernel<32><<<grid, 256, 0, st>>>(d_shards, h_hp->runs, *h_hp, epochs, step_now); break;
    case 64: runs_flush_kernel<64><<<grid, 256, 0, st>>>(d_shards, h_hp->runs, *h_hp, epochs, step_now); break;
    default: runs_flush_kernel<128><<<grid, 256, 0, st>>>(d_shards, h_hp->runs, *h_hp, epochs, step_now); break;
  }
  URE_CUDA(cudaGetLastError());
  return 0;
}
