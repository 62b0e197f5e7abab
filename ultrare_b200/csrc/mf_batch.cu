// Native host runtime of a K-shard training batch (the set-up half of Sisa.learn / Sisa.unlearn).
//
// The reference builds K models one after another in Python (method/sisa.py:33-36, 86-89 -> scratch.py:51-69).
// Here one call lays out EVERYTHING a batch needs inside one device allocation of the caller (weights, momentum,
// gradient scratch, losses, the owner schedule's sorted record copies, row offsets, radix scratch, schedule tables,
// the descriptor table, the training workspace), writes the descriptor table, clears what must be zero and queues
// the owner set-up kernels; a second call turns the plan those kernels leave into the launch parameters.  The host
// does no per-shard tensor bookkeeping before the training kernel is queued (round 1: ~0.5 ms of Python per step).
#include <string.h>

#include "common.cuh"

extern "C" int64_t ure_mf_train_workspace_bytes(void);
extern "C" int64_t ure_mf_owner_radix_bytes(int n_shards);
extern "C" int64_t ure_mf_owner_smem_bytes(int d, int cap_rows, int cap_slots, int cap_list, int spe_cap, int flags);
namespace ure {
int mf_owner_prepare_impl(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp, int epochs,
                          int max_rows, int32_t* d_radix_hist, void* d_workspace, void* stream, int flags);
}

static_assert(sizeof(ure_mf_batch_shard_t) == 32 && sizeof(ure_mf_batch_layout_t) == 152, "ctypes mirrors in _lib.py");

namespace ure {
namespace {
inline int64_t align_up(int64_t x) { return (x + 255) / 256 * 256; }
}  // namespace
}  // namespace ure

extern "C" int ure_mf_batch_layout(const ure_mf_batch_shard_t* h_shards, int n_shards, int n_item, int d, int batch,
                                   int epochs, int owner, int64_t sched_bytes_cap, ure_mf_batch_layout_t* out) {
  using namespace ure;
  URE_REQUIRE(h_shards && out && n_shards >= 1 && n_shards <= URE_MAX_SHARDS && n_item >= 1 && d >= 1 && batch >= 1,
              URE_EINVAL, "ure_mf_batch_layout: bad argument");
  memset(out, 0, sizeof(*out));
  int64_t rows = 0, n_tot = 0, n_off = 0, n_pinv = 0;
  int spe_cap = 1, max_rows = n_item, max_n = 0;
  for (int s = 0; s < n_shards; ++s) {
    URE_REQUIRE(h_shards[s].n >= 0 && h_shards[s].n_user >= 1, URE_EINVAL, "ure_mf_batch_layout: shard %d: n=%d n_user=%d",
                s, h_shards[s].n, h_shards[s].n_user);
    rows += h_shards[s].n_user;
    n_tot += h_shards[s].n;
    n_off += (int64_t)h_shards[s].n_user + n_item + 4;
    if (h_shards[s].perm) n_pinv += (int64_t)epochs * h_shards[s].n;
    const int spe = (h_shards[s].n + batch - 1) / batch;
    if (spe > spe_cap) spe_cap = spe;
    if (h_shards[s].n_user > max_rows) max_rows = h_shards[s].n_user;
    if (h_shards[s].n > max_n) max_n = h_shards[s].n;
  }
  const int grid = num_sms();
  const int64_t table_rows = rows + (int64_t)n_shards * n_item;
  int64_t o = 0;
  // the owner schedule wants the weights + momentum of every row in the SMs' shared memory: refuse cheaply
  const int64_t state = table_rows * 8 * d;
  out->owner = owner && n_shards <= grid && state <= (int64_t)grid * (200 << 10) && n_tot < (1ll << 31) && n_tot > 0;
  out->table = o; o = align_up(o + (int64_t)n_shards * sizeof(ure_mf_shard_t));
  out->W = o; o = align_up(o + table_rows * d * 4);
  // everything ure_mf_batch_setup clears is ONE region [ws, zero_end): workspace, momentum + scratch, losses, row offsets
  out->ws = o; o = align_up(o + ure_mf_train_workspace_bytes());
  out->Z = o; o = align_up(o + 2 * table_rows * d * 4);
  out->sse = o; o = align_up(o + (int64_t)n_shards * (epochs > 1 ? epochs : 1) * 8);
  int64_t n_rows = 0, stride = 0;
  if (out->owner) {
    out->off = o; o = align_up(o + n_off * 4);
    stride = 2 * n_tot > 0 ? 2 * n_tot : 1;
    const int64_t row_bytes = 2 * stride + 4ll * grid * (spe_cap + 1);
    n_rows = sched_bytes_cap / row_bytes;
    if (n_rows < 2) n_rows = 2;
    if (n_rows > epochs + 1) n_rows = epochs + 1;
  }
  out->zero_end = o;
  out->rows_total = rows;
  out->n_total = n_tot;
  out->spe_cap = spe_cap;
  out->max_rows = max_rows;
  out->max_n = max_n;
  out->grid = grid;
  if (out->owner) {
    out->rec = o; o = align_up(o + 4 * (n_tot > 0 ? n_tot : 1) * 16);
    out->radix = o; o = align_up(o + ure_mf_owner_radix_bytes(n_shards));
    out->perm_inv = o; o = align_up(o + n_pinv * 4);
    out->sched_rows = (int32_t)n_rows;
    out->sched_stride = stride;
    out->sched = o; o = align_up(o + n_rows * stride * 2);
    out->sched_off = o; o = align_up(o + n_rows * grid * (spe_cap + 1) * 4);
  }
  out->total = o;
  return 0;
}

extern "C" int ure_mf_batch_setup(const ure_mf_batch_shard_t* h_shards, int n_shards, int n_item,
                                  const ure_mf_hparams_t* h_hp, int epochs, uint32_t perm_seed, void* d_arena,
                                  const ure_mf_batch_layout_t* lay, void* h_stage, int flags, void* stream) {
  using namespace ure;
  URE_REQUIRE(h_shards && h_hp && d_arena && lay && h_stage, URE_EINVAL, "ure_mf_batch_setup: null argument");
  auto st = static_cast<cudaStream_t>(stream);
  char* const base = static_cast<char*>(d_arena);
  const int d = h_hp->d;
  const int E = epochs > 1 ? epochs : 1;
  auto* tab = static_cast<ure_mf_shard_t*>(h_stage);
  float* const W = reinterpret_cast<float*>(base + lay->W);
  float* const Z0 = reinterpret_cast<float*>(base + lay->Z);
  const int64_t table_rows = lay->rows_total + (int64_t)n_shards * n_item;
  float* const Z1 = Z0 + table_rows * d;
  int64_t prow = 0, r = 0, o = 0, pinv = 0;
  for (int s = 0; s < n_shards; ++s) {
    ure_mf_shard_t& t = tab[s];
    memset(&t, 0, sizeof(t));
    const int64_t qrow = lay->rows_total + (int64_t)s * n_item;
    t.inter = h_shards[s].inter;
    t.perm = h_shards[s].perm;
    t.P = W + prow * d;       t.Q = W + qrow * d;
    t.bufP = Z0 + prow * d;   t.bufQ = Z0 + qrow * d;
    t.gP = Z1 + prow * d;     t.gQ = Z1 + qrow * d;
    t.sse = reinterpret_cast<double*>(base + lay->sse) + (int64_t)s * E;
    t.n = h_shards[s].n; t.n_user = h_shards[s].n_user; t.n_item = n_item;
    t.shard_id = h_shards[s].shard_id; t.perm_seed = perm_seed; t.group = h_shards[s].group;
    if (lay->owner) {
      auto* rec = reinterpret_cast<ure_inter_t*>(base + lay->rec);
      const int64_t nt = lay->n_total > 0 ? lay->n_total : 1;
      t.inter_u = rec + r;          t.inter_i = rec + nt + r;
      t.tmp_u = rec + 2 * nt + r;   t.tmp_i = rec + 3 * nt + r;
      auto* off = reinterpret_cast<int32_t*>(base + lay->off);
      t.off_u = off + o;            t.off_i = off + o + t.n_user + 2;
      o += (int64_t)t.n_user + n_item + 4;
      if (t.perm) { t.perm_inv = reinterpret_cast<int32_t*>(base + lay->perm_inv) + pinv; pinv += (int64_t)epochs * t.n; }
      r += t.n;
    }
    prow += t.n_user;
  }
  URE_CUDA(cudaMemcpyAsync(base + lay->table, tab, (size_t)n_shards * sizeof(ure_mf_shard_t), cudaMemcpyHostToDevice, st));
  URE_CUDA(cudaMemsetAsync(base + lay->ws, 0, (size_t)(lay->zero_end - lay->ws), st));
  if (lay->owner) {
    bool any_perm = false;
    for (int s = 0; s < n_shards; ++s) any_perm |= h_shards[s].perm != nullptr;
    const bool no_plan = (flags & URE_BATCH_NO_PLAN) != 0;
    // 1: the workspace has just been cleared | 2: no plan kernel | 4: no explicit visiting orders to invert | 8: the
    // set-up of a small batch is launch-bound: one cooperative launch (owner_setup_kernel) instead of eight
    if (int rc = mf_owner_prepare_impl(reinterpret_cast<const ure_mf_shard_t*>(base + lay->table), n_shards, h_hp, epochs,
                                       lay->max_rows, reinterpret_cast<int32_t*>(base + lay->radix), base + lay->ws, stream,
                                       1 | (no_plan ? 2 : 0) | (any_perm ? 0 : 4) | (lay->n_total <= (8ll << 20) ? 8 : 0)))
      return rc;
    // the plan (4 ints) travels to the page-locked block right behind the descriptor table
    if (!no_plan)
      URE_CUDA(cudaMemcpyAsync(static_cast<char*>(h_stage) + (size_t)n_shards * sizeof(ure_mf_shard_t), base + lay->ws, 16,
                               cudaMemcpyDeviceToHost, st));
  }
  return 0;
}

extern "C" int ure_mf_batch_plan(const int32_t* h_plan, int n_shards, ure_mf_hparams_t* hp, void* d_arena,
                                 const ure_mf_batch_layout_t* lay, int allow_cache, int force_flags, int force_list,
                                 int32_t* h_info) {
  using namespace ure;
  URE_REQUIRE(h_plan && hp && d_arena && lay, URE_EINVAL, "ure_mf_batch_plan: null argument");
  if (!lay->owner) return 0;
  const int max_rows = h_plan[0], max_slots = h_plan[1], max_spe = h_plan[2], avail = h_plan[3];
  const int cap_rows = max_rows > 1 ? max_rows : 1;
  int cap_slots = (max_slots + 15) / 16 * 16;
  if (cap_slots < 16) cap_slots = 16;
  const int spe_cap = max_spe > 1 ? max_spe : 1;
  const int d = hp->d;
  auto need_of = [&](int cap_list, int flags) {
    return (long long)ure_mf_owner_smem_bytes(d, cap_rows, cap_slots, cap_list, spe_cap, flags);
  };
  // shared-memory configurations, fastest first: record cache (every owned slot's record resident); batch lists and
  // their records staged per step, as many entries as fit (a longer list is read from the schedule table); the same
  // with the schedule pre-pass running without its record-index cache
  int flags = -1, cap_list = cap_slots;
  if (force_flags >= 0) {
    flags = force_flags;
    cap_list = force_list / 16 * 16;
    if (cap_list < 16) cap_list = 16;
    if (cap_list > cap_slots) cap_list = cap_slots;
    if (need_of(cap_list, flags) > avail) flags = -1;
  } else {
    if (allow_cache && lay->max_rows <= (1 << 20) && need_of(cap_slots, 1) <= avail) { flags = 1; cap_list = cap_slots; }
    for (int f = 0; flags < 0 && f <= 2; f += 2) {
      const long long need16 = need_of(16, f);
      if (need16 > avail) continue;
      long long c = 16 + (avail - need16) / 160 * 16;            // 10 bytes of shared memory per staged entry
      if (c > cap_slots) c = cap_slots;
      if (need_of((int)c, f) <= avail && c >= (cap_slots < 1024 ? cap_slots : 1024)) { flags = f; cap_list = (int)c; }
    }
  }
  const bool fits = flags >= 0 && cap_slots <= 65520 && cap_rows < 4096 && max_spe <= 8192;
  if (h_info) {
    h_info[0] = fits; h_info[1] = flags; h_info[2] = cap_list; h_info[3] = cap_rows; h_info[4] = cap_slots;
    h_info[5] = spe_cap; h_info[6] = flags >= 0 ? (int)need_of(cap_list, flags) : 0; h_info[7] = avail;
  }
  if (!fits) return 0;
  char* const base = static_cast<char*>(d_arena);
  hp->mode = URE_MF_OWNER;
  hp->owner_cap_rows = cap_rows; hp->owner_cap_slots = cap_slots; hp->owner_spe_cap = spe_cap;
  hp->owner_flags = flags; hp->owner_cap_list = cap_list;
  hp->owner_sched = reinterpret_cast<uint16_t*>(base + lay->sched);
  hp->owner_sched_off = reinterpret_cast<int32_t*>(base + lay->sched_off);
  hp->owner_sched_rows = lay->sched_rows; hp->owner_sched_stride = lay->sched_stride; hp->owner_sched_step0 = 0;
  hp->owner_max_n = lay->max_n;
  // the offsets table was laid out for the host-side steps-per-epoch bound; the plan's is the same number
  URE_REQUIRE(spe_cap <= lay->spe_cap, URE_EINVAL, "ure_mf_batch_plan: plan steps per epoch %d above the layout's %d",
              spe_cap, lay->spe_cap);
  hp->owner_spe_cap = lay->spe_cap;
  return 1;
}
