// Fused Matrix-Factorization training step for ALL shard models in one persistent launch.
//
// Replaces the body of baseTrain (reference method/utils.py:58-98): per batch
//   pred = sum_t P[u,t]*Q[i,t]; e = pred - r; L += e^2;
//   gP[u] += 2e*Q[i]; gQ[i] += 2e*P[u]            (all with PRE-step weights)
// followed by the dense optim.SGD(momentum, weight_decay) update of scratch.py:65-68
// on every row of both tables, for every shard (the K sequential Scratch.train calls
// of method/sisa.py:33-36,86-89 become one launch).
//
// One cooperative launch, one CTA per SM, all steps inside.  The batch-synchronous semantics
// need two grid-wide barriers per step; on this 148-SM part a barrier costs ~2 us of pure
// latency, so each barrier is split into ARRIVE and WAIT and everything that does not depend
// on the other CTAs is issued in between:
//
//   gradients(t)   gather P[u], Q[i] (16-byte L2 loads), shuffle dot product, loss,
//                  red.global.add.v4.f32 scatter of both gradient rows -- INTO THE MOMENTUM ARRAYS, which
//                  between two sweeps hold pre = mu*buf + wd*w, so that pre + sum(g) is the new momentum:
//                  no gradient arrays, the sweep moves 4 instead of 6 table-sized streams
//   ARRIVE 1       -- overlap: load this thread's sweep operand w (unchanged by the gradient phase);
//                     warp 1 builds the step tables of t+1
//   WAIT 1
//   sweep(t)       dense SGD on every row of every active shard: buf = pre + sum(g) (already in memory);
//                  w -= lr*buf; pre' = mu*buf + wd*w  (the true buf at a shard's last step of the launch)
//   ARRIVE 2       -- overlap: permutation index + record fetch of this warp's chunk of t+1
//   WAIT 2
//
// The visiting order is either an explicit permutation (parity runs against the reference) or
// the inline Feistel permutation (feistel.cuh).
//
// The same schedule trains the BPR objective (ure_mf_train_bpr, LOSS = kBpr): the lane that fetches record idx also
// draws its negative j (bpr_sampler.cuh) from the user's seen list; with x = P[u].(Q[i] - Q[j]) and c = sigmoid(-x)
// the triple adds softplus(-x) to the loss and scatters -c (Q[i] - Q[j]) into row u, -c P[u] into row i and
// +c P[u] into row j (three REDs, PRE-step weights).  A dropped triple (j = -1) adds nothing.
//
// This header holds the schedule; mf_train.cu instantiates it for MSE (ure_mf_train), bpr.cu for BPR
// (ure_mf_train_bpr).  The two objectives live in separate translation units so that adding one leaves the
// other's machine code as it was.
#pragma once
#include "bpr_sampler.cuh"
#include "common.cuh"
#include "feistel.cuh"

namespace ure {

extern int g_force_warps_g0;   // diagnostics (ure_mf_debug_flags bits 8..13): force the warp split, 32 = one group

namespace {

constexpr int kThreads = 1024;
constexpr int KM = URE_MAX_SHARDS;
constexpr int kMse = 0, kBpr = 1;     // training objective (template parameter LOSS)

struct Workspace {
  unsigned barrier[2];     // one monotonic counter per warp group
  long long* trace;        // optional [steps][gridDim.x][6] SM-clock stamps (ure_mf_train_trace), else NULL
  int trace_steps;
  unsigned debug_flags;    // diagnostics only: 1 = skip gradient REDs, 2 = identity visiting order
  unsigned pad[58];
};
static_assert(sizeof(Workspace) == 256, "workspace layout");

struct ShardPtrs {         // 32 bytes: fetched with two LDS.128
  float* P; float* Q; float* gP; float* gQ;
};

// Step tables, double buffered (built for t+1 while step t is still running).
struct StepTables {
  int item_prefix[KM + 1];           // flattened batch positions of the active shards
  long long row_prefix[2 * KM + 1];  // flattened float4 elements of the dense sweep
  int epoch[KM];                     // -1: shard finished
  int start[KM];                     // first position of the batch inside the epoch
  float lr[KM];
  FeistelKeys keys[KM];
  unsigned char last[KM];            // 1: the shard's last step of this launch (its momentum is stored as such)
};

// BPR only: per-launch constants of the sampler, in dynamic shared memory after the four StepTables (the MSE
// instantiations neither allocate nor touch it).  key[b][s] = perm_key of shard s's epoch in step-table buffer b.
struct BprSmem {
  uint32_t key[4][KM];
  const int64_t* seen_off[KM];
  const int32_t* seen_items[KM];
};
__device__ __forceinline__ BprSmem* bpr_smem(unsigned char* dyn) {
  return reinterpret_cast<BprSmem*>(dyn + 4 * sizeof(StepTables));
}

// largest s with prefix[s] <= x  (prefix[0] = 0, prefix[nseg] = total > x)
template <typename T>
__device__ __forceinline__ int find_segment(const T* prefix, int nseg, T x) {
  int lo = 0, hi = nseg;
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (prefix[mid] <= x) lo = mid; else hi = mid;
  }
  return lo;
}

// ---- split grid barrier (monotonic counter; cooperative launch guarantees co-residency).
// A CTA hosts up to two independent warp groups; each group synchronises on its own named barrier
// (bar.sync id, count) and its own global counter, so a group waiting at a grid barrier leaves the SM to
// the other group's warps.
__device__ __forceinline__ void group_sync(int bar_id, int n_threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(n_threads) : "memory");
}
__device__ __forceinline__ void barrier_arrive(unsigned* counter, int bar_id, int n_threads, bool leader) {
  group_sync(bar_id, n_threads);          // every warp of the group has issued its writes / REDs
  if (leader) {
    __threadfence();                      // cumulative: orders the group's prior writes before the arrival
    atomicAdd(counter, 1u);
  }
}
__device__ __forceinline__ void barrier_wait(unsigned* counter, unsigned target, int bar_id, int n_threads,
                                             bool leader) {
  if (leader) {
    while (*reinterpret_cast<volatile unsigned*>(counter) < target) {
    }
    __threadfence();
  }
  group_sync(bar_id, n_threads);
}

// Gradient work of one 32-interaction warp chunk.  Lane l fetched interaction l (u, it, r, shard s or -1);
// a group of G = D/4 lanes processes its G interactions SUB at a time (2*SUB 16-byte gathers in flight).
// UNIFORM: the whole chunk lies in shard tables `tp`; otherwise each interaction looks its shard up.
// BPR: the record's rating is not used; `r` carries the bits of its negative j instead (fetch), -1 = dropped.
// Returns the error e of the lane's interaction (MSE), or its loss softplus(-x) (BPR; 0 for a dropped triple).
template <int D, bool UNIFORM, int LOSS>
__device__ __forceinline__ float chunk_gradients(int u, int it, float r, int s, const ShardPtrs& tp,
                                                  const ShardPtrs* s_ptr, int gl, unsigned dbg) {
  constexpr int G = D / 4;
  if constexpr (LOSS == kBpr) {
    // three gathered rows per triple: one triple per lane group at a time fits __launch_bounds__(1024, 1) without
    // spills (two in flight spill 8 / 44 / 12 bytes at d = 32 / 64 / 128)
    constexpr int SUB = 1;
    float my_l = 0.f;
#pragma unroll
    for (int q0 = 0; q0 < G; q0 += SUB) {
      float4 pu[SUB], qd[SUB];
      int uq[SUB], iq[SUB], jq[SUB], sq[SUB];
#pragma unroll
      for (int q = 0; q < SUB; ++q) {
        uq[q] = __shfl_sync(0xffffffffu, u, q0 + q, G);
        iq[q] = __shfl_sync(0xffffffffu, it, q0 + q, G);
        jq[q] = __shfl_sync(0xffffffffu, __float_as_int(r), q0 + q, G);
        sq[q] = __shfl_sync(0xffffffffu, s, q0 + q, G);
        if (jq[q] < 0) sq[q] = -1;               // dropped triple: no loss, no gradient
        pu[q] = make_float4(0.f, 0.f, 0.f, 0.f);
        qd[q] = pu[q];
        if (sq[q] >= 0) {
          const float* Pb = UNIFORM ? tp.P : s_ptr[sq[q]].P;
          const float* Qb = UNIFORM ? tp.Q : s_ptr[sq[q]].Q;
          pu[q] = ld_cg_f4(Pb + (size_t)uq[q] * D + 4 * gl);
          const float4 qi = ld_cg_f4(Qb + (size_t)iq[q] * D + 4 * gl);
          const float4 qj = ld_cg_f4(Qb + (size_t)jq[q] * D + 4 * gl);
          qd[q] = make_float4(qi.x - qj.x, qi.y - qj.y, qi.z - qj.z, qi.w - qj.w);
        }
      }
#pragma unroll
      for (int q = 0; q < SUB; ++q) {
        float x = pu[q].x * qd[q].x;
        x = fmaf(pu[q].y, qd[q].y, x);
        x = fmaf(pu[q].z, qd[q].z, x);
        x = fmaf(pu[q].w, qd[q].w, x);
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o, G);
        // softplus(-x) = max(-x, 0) + log1p(exp(-|x|)); sigmoid(-x) = 1 / (1 + exp(x))
        const float l = fmaxf(-x, 0.f) + log1pf(expf(-fabsf(x)));
        if (gl == q0 + q && sq[q] >= 0) my_l = l;
        if (sq[q] >= 0 && !(dbg & 1u)) {
          float* gPb = UNIFORM ? tp.gP : s_ptr[sq[q]].gP;
          float* gQb = UNIFORM ? tp.gQ : s_ptr[sq[q]].gQ;
          const float c = 1.f / (1.f + expf(x));
          red_add_f4(gPb + (size_t)uq[q] * D + 4 * gl, -c * qd[q].x, -c * qd[q].y, -c * qd[q].z, -c * qd[q].w);
          red_add_f4(gQb + (size_t)iq[q] * D + 4 * gl, -c * pu[q].x, -c * pu[q].y, -c * pu[q].z, -c * pu[q].w);
          red_add_f4(gQb + (size_t)jq[q] * D + 4 * gl, c * pu[q].x, c * pu[q].y, c * pu[q].z, c * pu[q].w);
        }
      }
    }
    return my_l;
  }
  constexpr int SUB = (G < 4) ? G : 4;
  float my_e = 0.f;
#pragma unroll
  for (int q0 = 0; q0 < G; q0 += SUB) {
    float4 pu[SUB], qi[SUB];
    int uq[SUB], iq[SUB], sq[SUB];
    float rq[SUB];
#pragma unroll
    for (int q = 0; q < SUB; ++q) {
      uq[q] = __shfl_sync(0xffffffffu, u, q0 + q, G);
      iq[q] = __shfl_sync(0xffffffffu, it, q0 + q, G);
      rq[q] = __shfl_sync(0xffffffffu, r, q0 + q, G);
      sq[q] = __shfl_sync(0xffffffffu, s, q0 + q, G);
      pu[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      qi[q] = pu[q];
      if (sq[q] >= 0) {
        const float* Pb = UNIFORM ? tp.P : s_ptr[sq[q]].P;
        const float* Qb = UNIFORM ? tp.Q : s_ptr[sq[q]].Q;
        pu[q] = ld_cg_f4(Pb + (size_t)uq[q] * D + 4 * gl);
        qi[q] = ld_cg_f4(Qb + (size_t)iq[q] * D + 4 * gl);
      }
    }
#pragma unroll
    for (int q = 0; q < SUB; ++q) {
      float dot = pu[q].x * qi[q].x;
      dot = fmaf(pu[q].y, qi[q].y, dot);
      dot = fmaf(pu[q].z, qi[q].z, dot);
      dot = fmaf(pu[q].w, qi[q].w, dot);
#pragma unroll
      for (int o = G / 2; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o, G);
      const float e = dot - rq[q];
      if (gl == q0 + q) my_e = e;
      if (sq[q] >= 0 && !(dbg & 1u)) {
        float* gPb = UNIFORM ? tp.gP : s_ptr[sq[q]].gP;
        float* gQb = UNIFORM ? tp.gQ : s_ptr[sq[q]].gQ;
        const float ge = 2.f * e;
        red_add_f4(gPb + (size_t)uq[q] * D + 4 * gl, ge * qi[q].x, ge * qi[q].y, ge * qi[q].z, ge * qi[q].w);
        red_add_f4(gQb + (size_t)iq[q] * D + 4 * gl, ge * pu[q].x, ge * pu[q].y, ge * pu[q].z, ge * pu[q].w);
      }
    }
  }
  return my_e;
}

// Shards never interact, so the CTA's 32 warps are split into (up to) two warp GROUPS, each running the
// whole step pipeline for its own subset of the shards (ure_mf_shard_t::group) with its own named barrier
// and its own grid-barrier counter: while one group sits in a barrier, the SM executes the other's warps.
template <int D, int LOSS>
__global__ void __launch_bounds__(kThreads, 1)
mf_train_kernel(const ure_mf_shard_t* __restrict__ shards, int K, ure_mf_hparams_t hp, int epochs,
                long long step_begin, long long step_end, Workspace* ws, int warps_g0,
                const ure_bpr_shard_t* __restrict__ bpr) {
  constexpr int G = D / 4;                 // lanes per interaction
  // ---- per-CTA shard tables (static shared memory): constant for the whole launch
  __shared__ ShardPtrs s_ptr[KM];
  __shared__ const ure_inter_t* s_inter[KM];
  __shared__ const int32_t* s_perm[KM];
  __shared__ float* s_buf[2 * KM];         // bufP, bufQ
  __shared__ double* s_sse[KM];
  __shared__ int s_n[KM], s_nuser[KM], s_nitem[KM], s_spe[KM], s_shard_id[KM];
  __shared__ unsigned char s_group[KM];
  __shared__ uint32_t s_seed[KM];
  __shared__ FeistelDomain s_dom[KM];
  // ---- per-shard schedule cursor (advanced by the table builder) and the double-buffered step tables
  __shared__ int s_cur_epoch[KM], s_cur_batch[KM];
  extern __shared__ __align__(16) unsigned char dyn_smem[];     // StepTables[2 groups][2] (static limit is 48 KB), BPR: + BprSmem
  StepTables* const s_tab_all = reinterpret_cast<StepTables*>(dyn_smem);
  __shared__ float s_sse_acc[KM];

  const int lane = threadIdx.x & 31;
  const int gl = lane % G;
  for (int s = threadIdx.x; s < K; s += kThreads) {
    const ure_mf_shard_t sh = shards[s];
    s_ptr[s] = ShardPtrs{sh.P, sh.Q, sh.bufP, sh.bufQ};      // gradients are reduced into the momentum arrays
    s_inter[s] = sh.inter; s_perm[s] = sh.perm;
    s_buf[2 * s] = sh.bufP; s_buf[2 * s + 1] = sh.bufQ;
    s_sse[s] = sh.sse;
    s_n[s] = sh.n; s_nuser[s] = sh.n_user; s_nitem[s] = sh.n_item;
    const int spe = (sh.n + hp.batch - 1) / hp.batch;
    s_spe[s] = spe;
    s_seed[s] = sh.perm_seed; s_shard_id[s] = sh.shard_id;
    s_group[s] = (unsigned char)((warps_g0 < kThreads / 32) ? (sh.group & 1) : 0);
    s_dom[s].init((uint32_t)sh.n);
    s_cur_epoch[s] = spe > 0 ? (int)(step_begin / spe) : epochs;     // the only divisions of the launch
    s_cur_batch[s] = spe > 0 ? (int)(step_begin % spe) : 0;
    s_sse_acc[s] = 0.f;
    if constexpr (LOSS == kBpr) {
      bpr_smem(dyn_smem)->seen_off[s] = bpr[s].seen_off;
      bpr_smem(dyn_smem)->seen_items[s] = bpr[s].seen_items;
    }
  }
  __syncthreads();

  // ---- this thread's warp group
  const int grp = (int)(threadIdx.x >> 5) < warps_g0 ? 0 : 1;
  const int g_warps = grp == 0 ? warps_g0 : kThreads / 32 - warps_g0;     // warps of the group in this CTA
  const int g_threads = g_warps * 32;
  const int tid = threadIdx.x - (grp == 0 ? 0 : warps_g0 * 32);          // thread index inside the group
  const int warp = tid >> 5;
  const int bar_id = grp + 1;                                             // named barrier of the group
  const bool leader = tid == 0;
  unsigned* const counter = &ws->barrier[grp];
  StepTables* const s_tab = s_tab_all + 2 * grp;
  const unsigned dbg = ws->debug_flags;
  long long* const trace = ws->trace;
  const int trace_steps = ws->trace_steps;
  const long long n_threads = (long long)gridDim.x * g_threads;          // the group's threads grid-wide
  const long long gtid = (long long)blockIdx.x * g_threads + tid;
  const int n_warps = (int)(n_threads >> 5);
  // chunk index of this warp: CTA-minor, so that a step with fewer chunks than warps still uses every SM
  const int gwarp = warp * (int)gridDim.x + (int)blockIdx.x;
  const float wd = hp.weight_decay, mu = hp.momentum;
  unsigned bar_target = 0;

  // Step tables of the group for the step its shards' cursors point at, then advance the cursors.  Executed
  // by ONE warp (lanes = shards, 32 at a time, prefix carried): no block-wide synchronisation inside.
  auto build_tables = [&](StepTables& tb, long long t_build) {
    int carry = 0;
    long long carry2 = 0;
    for (int base = 0; base < K; base += 32) {
      const int s = base + lane;
      int cnt = 0, ep = -1, st = 0;
      long long rows_u = 0, rows_i = 0;
      if (s < K && s_group[s] == grp) {
        const int spe = s_spe[s];
        ep = s_cur_epoch[s];
        const int bi = s_cur_batch[s];
        if (spe > 0 && ep < epochs) {
          st = bi * hp.batch;
          cnt = min(hp.batch, s_n[s] - st);
          rows_u = (long long)s_nuser[s] * G;
          rows_i = (long long)s_nitem[s] * G;
          double lr = (double)hp.lr0;
          for (int q = ep / hp.lr_step; q > 0; --q) lr *= (double)hp.lr_decay;
          tb.lr[s] = (float)lr;
          tb.keys[s].init(perm_key(s_seed[s], (uint32_t)s_shard_id[s], (uint32_t)ep));
          if constexpr (LOSS == kBpr)
            bpr_smem(dyn_smem)->key[&tb - s_tab_all][s] = perm_key(s_seed[s], (uint32_t)s_shard_id[s], (uint32_t)ep);
          tb.last[s] = (unsigned char)((bi + 1 == spe && ep + 1 == epochs) || t_build + 1 == step_end);
          if (bi + 1 == spe) { s_cur_epoch[s] = ep + 1; s_cur_batch[s] = 0; }
          else s_cur_batch[s] = bi + 1;
        } else {
          ep = -1;
        }
      }
      if (s < K) {
        tb.epoch[s] = ep;
        tb.start[s] = st;
      }
      int v = cnt;
      long long v2 = rows_u + rows_i;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int a = __shfl_up_sync(0xffffffffu, v, o);
        const long long b = __shfl_up_sync(0xffffffffu, v2, o);
        if (lane >= o) { v += a; v2 += b; }
      }
      if (s < K) {
        tb.item_prefix[s + 1] = v + carry;
        tb.row_prefix[2 * s + 1] = v2 + carry2 - rows_i;
        tb.row_prefix[2 * s + 2] = v2 + carry2;
      }
      carry += __shfl_sync(0xffffffffu, v, 31);
      carry2 += __shfl_sync(0xffffffffu, v2, 31);
    }
    if (lane == 0) { tb.item_prefix[0] = 0; tb.row_prefix[0] = 0; }
  };

  // Visiting-order index + record of this lane's interaction in warp chunk `wc` of the step in `tb` (and, BPR, the
  // record's negative: bpr_sampler.cuh, keyed like the epoch's visiting order).
  auto fetch = [&](const StepTables& tb, int wc, int& s, int& u, int& it, float& r) {
    const int item = wc * 32 + lane;
    s = -1; u = 0; it = 0; r = 0.f;
    if (item < tb.item_prefix[K]) {
      s = find_segment(tb.item_prefix, K, item);
      const int j = tb.start[s] + (item - tb.item_prefix[s]);
      const int32_t* pm = s_perm[s];
      uint32_t idx;
      if (pm) idx = (uint32_t)__ldg(pm + (long long)tb.epoch[s] * s_n[s] + j);
      else if (dbg & 2u) idx = (uint32_t)j;
      else idx = feistel(s_dom[s], tb.keys[s], (uint32_t)j);
      const int4 rec = ld_stream_i4(s_inter[s] + idx);
      u = rec.x; it = rec.y; r = __int_as_float(rec.z);
      if constexpr (LOSS == kBpr) {
        const BprSmem* b = bpr_smem(dyn_smem);
        const int64_t* off = b->seen_off[s];
        r = __int_as_float(bpr_negative(b->key[&tb - s_tab_all][s], idx, b->seen_items[s], __ldg(off + u),
                                        __ldg(off + u + 1), (uint32_t)s_nitem[s]));
      }
    }
  };

#define URE_STAMP(PH)                                                                                  \
  if (trace && leader && grp == 0 && (t - step_begin) < trace_steps)                                   \
    trace[((t - step_begin) * gridDim.x + blockIdx.x) * 6 + (PH)] = clock64();

  // ---- prologue: tables and first-chunk records of the group's first step
  if (warp == 0) build_tables(s_tab[0], step_begin);
  group_sync(bar_id, g_threads);
  int ps, pu_, pi_;
  float pr_;
  fetch(s_tab[0], gwarp, ps, pu_, pi_, pr_);
  // the momentum arrays of the shards that train in this launch: buf -> pre = mu*buf + wd*w, then a grid barrier
  // before the first gradients are reduced into them
  if (step_begin < step_end) {
    const StepTables& tb = s_tab[0];
    const long long total4 = tb.row_prefix[2 * K];
    for (long long x = gtid; x < total4; x += n_threads) {
      const int seg = find_segment(tb.row_prefix, 2 * K, x);
      const size_t off = (size_t)(x - tb.row_prefix[seg]) * 4;
      const ShardPtrs tq = s_ptr[seg >> 1];
      const float4 w = ld_cg_f4(((seg & 1) ? tq.Q : tq.P) + off);
      float4 b = ld_cg_f4(s_buf[seg] + off);
      b.x = fmaf(mu, b.x, __fmul_rn(wd, w.x)); b.y = fmaf(mu, b.y, __fmul_rn(wd, w.y));
      b.z = fmaf(mu, b.z, __fmul_rn(wd, w.z)); b.w = fmaf(mu, b.w, __fmul_rn(wd, w.w));
      st_cg_f4(s_buf[seg] + off, b);
    }
    barrier_arrive(counter, bar_id, g_threads, leader);
    bar_target += gridDim.x;
    barrier_wait(counter, bar_target, bar_id, g_threads, leader);
  }

  int cur = 0;
  for (long long t = step_begin; t < step_end; ++t, cur ^= 1) {
    const StepTables& tb = s_tab[cur];
    const bool more = t + 1 < step_end;
    URE_STAMP(0)
    // ---------------------------------------------------------------- gradients
    const int total = tb.item_prefix[K];
    float acc = 0.f;          // sum of e^2 of the chunks this warp processed, all in shard acc_s
    int acc_s = -1;
    for (int wc = gwarp; wc * 32 < total; wc += n_warps) {
      int s, u, it;
      float r;
      if (wc == gwarp) { s = ps; u = pu_; it = pi_; r = pr_; }      // prefetched behind WAIT 2 of step t-1
      else fetch(tb, wc, s, u, it, r);
      const bool valid = s >= 0;
      // the common case: the whole 32-interaction chunk lies in one shard -> table pointers once per warp
      const int s0 = __shfl_sync(0xffffffffu, s, 0);
      const bool uniform = __all_sync(0xffffffffu, s == s0 || !valid);
      const ShardPtrs tp = s_ptr[s0];
      const float my_e = uniform ? chunk_gradients<D, true, LOSS>(u, it, r, s, tp, s_ptr, gl, dbg)
                                 : chunk_gradients<D, false, LOSS>(u, it, r, s, tp, s_ptr, gl, dbg);
      // loss: warp-reduce when the chunk is single-shard (one shared atomic per warp, not per lane)
      const float e2 = valid ? (LOSS == kBpr ? my_e : my_e * my_e) : 0.f;
      if (uniform) {
        const float w = warp_sum(e2);
        if (s0 != acc_s) {
          if (acc_s >= 0 && lane == 0) atomicAdd(&s_sse_acc[acc_s], acc);
          acc = 0.f;
          acc_s = s0;
        }
        acc += w;                                   // every lane carries the warp total; lane 0 publishes
      } else if (valid) {
        atomicAdd(&s_sse_acc[s], e2);
      }
    }
    if (acc_s >= 0 && lane == 0) atomicAdd(&s_sse_acc[acc_s], acc);
    URE_STAMP(1)
    barrier_arrive(counter, bar_id, g_threads, leader);     // ---------------- ARRIVE 1
    bar_target += gridDim.x;
    // overlap: publish the loss, preload the sweep operands that the gradient phase did not touch,
    // build the tables of step t+1
    for (int s = tid; s < K; s += g_threads) {
      if (s_group[s] != grp) continue;
      const float v = s_sse_acc[s];
      if (v != 0.f) {
        atomicAdd(s_sse[s] + tb.epoch[s], (double)v);
        s_sse_acc[s] = 0.f;
      }
    }
    const long long total4 = tb.row_prefix[2 * K];
    int seg0 = 0;
    size_t off0 = 0;
    float4 w0 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (gtid < total4) {
      seg0 = find_segment(tb.row_prefix, 2 * K, gtid);
      off0 = (size_t)(gtid - tb.row_prefix[seg0]) * 4;
      const ShardPtrs tp = s_ptr[seg0 >> 1];
      w0 = ld_cg_f4(((seg0 & 1) ? tp.Q : tp.P) + off0);
    }
    if (warp == (g_warps > 1 ? 1 : 0) && more) build_tables(s_tab[cur ^ 1], t + 1);
    URE_STAMP(2)
    barrier_wait(counter, bar_target, bar_id, g_threads, leader);   // -------- WAIT 1
    URE_STAMP(3)

    // ---------------------------------------------------------------- dense SGD sweep
    for (long long x = gtid; x < total4; x += n_threads) {
      int seg;
      size_t off;
      float4 w;
      if (x == gtid) { seg = seg0; off = off0; w = w0; }
      else {
        seg = find_segment(tb.row_prefix, 2 * K, x);
        off = (size_t)(x - tb.row_prefix[seg]) * 4;
        const ShardPtrs tq = s_ptr[seg >> 1];
        w = ld_cg_f4(((seg & 1) ? tq.Q : tq.P) + off);
      }
      const ShardPtrs tp = s_ptr[seg >> 1];
      float* W = (seg & 1) ? tp.Q : tp.P;
      float* Bf = s_buf[seg];
      const float nlr = -tb.lr[seg >> 1];
      // torch SGD: buf = buf*mu + (g + wd*w) -- here pre + sum(g), already reduced in memory; w = w + (-lr)*buf
      float4 b = ld_cg_f4(Bf + off);
      w.x = fmaf(nlr, b.x, w.x); w.y = fmaf(nlr, b.y, w.y); w.z = fmaf(nlr, b.z, w.z); w.w = fmaf(nlr, b.w, w.w);
      st_cg_f4(W + off, w);
      if (!tb.last[seg >> 1]) {             // next step's pre; the true momentum at the shard's last step
        b.x = fmaf(mu, b.x, __fmul_rn(wd, w.x)); b.y = fmaf(mu, b.y, __fmul_rn(wd, w.y));
        b.z = fmaf(mu, b.z, __fmul_rn(wd, w.z)); b.w = fmaf(mu, b.w, __fmul_rn(wd, w.w));
        st_cg_f4(Bf + off, b);
      }
    }
    URE_STAMP(4)
    barrier_arrive(counter, bar_id, g_threads, leader);     // ---------------- ARRIVE 2
    bar_target += gridDim.x;
    // overlap: visiting-order index + record of this warp's first chunk of step t+1 (static data);
    // the tables of t+1 were written before WAIT 1's group barrier
    if (more) fetch(s_tab[cur ^ 1], gwarp, ps, pu_, pi_, pr_);
    barrier_wait(counter, bar_target, bar_id, g_threads, leader);   // -------- WAIT 2
    URE_STAMP(5)
  }
#undef URE_STAMP
}

template <int D, int LOSS>
int launch(const ure_mf_shard_t* d_shards, int K, const ure_mf_hparams_t& hp, int epochs, long long s0,
           long long s1, Workspace* ws, int warps_g0, const ure_bpr_shard_t* bpr, cudaStream_t st) {
  auto kern = mf_train_kernel<D, LOSS>;
  const size_t smem = 4 * sizeof(StepTables) + (LOSS == kBpr ? sizeof(BprSmem) : 0);
  URE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  URE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kThreads, smem));
  URE_REQUIRE(occ >= 1, URE_ECOOP, "mf_train_kernel<%d> cannot be resident", D);
  const int grid = num_sms();
  if (g_force_warps_g0 >= 1 && g_force_warps_g0 <= 32) warps_g0 = g_force_warps_g0;
  URE_CUDA(cudaMemsetAsync(ws->barrier, 0, 2 * sizeof(unsigned), st));
  void* args[] = {(void*)&d_shards, (void*)&K,  (void*)&hp,       (void*)&epochs,
                  (void*)&s0,       (void*)&s1, (void*)&ws,       (void*)&warps_g0, (void*)&bpr};
  URE_CUDA(cudaLaunchCooperativeKernel((void*)kern, dim3(grid), dim3(kThreads), args, smem, st));
  return 0;
}

template <int LOSS>
int dense(const ure_mf_shard_t* d_shards, int K, const ure_mf_hparams_t& hp, int epochs, long long s0, long long s1,
          int warps_g0, void* d_workspace, const ure_bpr_shard_t* bpr, void* stream, const char* who) {
  if (s1 <= s0) return 0;
  auto* ws = static_cast<Workspace*>(d_workspace);
  auto st = static_cast<cudaStream_t>(stream);
  switch (hp.d) {
    case 8: return launch<8, LOSS>(d_shards, K, hp, epochs, s0, s1, ws, warps_g0, bpr, st);
    case 16: return launch<16, LOSS>(d_shards, K, hp, epochs, s0, s1, ws, warps_g0, bpr, st);
    case 32: return launch<32, LOSS>(d_shards, K, hp, epochs, s0, s1, ws, warps_g0, bpr, st);
    case 64: return launch<64, LOSS>(d_shards, K, hp, epochs, s0, s1, ws, warps_g0, bpr, st);
    case 128: return launch<128, LOSS>(d_shards, K, hp, epochs, s0, s1, ws, warps_g0, bpr, st);
    default:
      set_error("%s: d=%d not in {8,16,32,64,128}", who, hp.d);
      return URE_EUNSUPPORTED;
  }
}

}  // namespace
}  // namespace ure
