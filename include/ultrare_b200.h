/*
 * ultrare_b200 -- C ABI of the B200-native UltraRE sharded-retraining hot path.
 *
 * The reference (ZhangYizhao/UltraRE) has no FFI layer: its seam is the Python
 * call surface of method/utils.py, method/scratch.py, method/sisa.py, group.py
 * (SURVEY.md §8b).  Each entry point below replaces the arithmetic of one of
 * those Python functions; the reference-side binding is a ctypes stub
 * (INTEGRATION.md).  Conventions:
 *   - every pointer is a raw DEVICE address unless its name starts with h_;
 *     the caller (PyTorch) owns all memory, the library allocates nothing that
 *     outlives a call;
 *   - every launch is asynchronous on the caller's `stream` (a cudaStream_t cast
 *     to void*); the library never synchronises;
 *   - every function returns 0 on success, a positive cudaError_t or a negative
 *     URE_E* code otherwise; ure_last_error() gives the thread-local message;
 *   - indices are int32 on device; interactions are packed 16-byte records.
 */
#ifndef ULTRARE_B200_H
#define ULTRARE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define URE_ABI_VERSION 7
#define URE_MAX_SHARDS 256        /* shard models batched in one launch           */
#define URE_TOP_K 10              /* baseTest(top_k=10), method/utils.py:115      */

#define URE_EINVAL (-1)           /* bad argument                                  */
#define URE_EUNSUPPORTED (-2)     /* shape outside what the kernels are built for  */
#define URE_ECOOP (-3)            /* cooperative launch cannot be made resident    */

/* One rating: what RatingData.__getitem__ yields (read.py:118-124) --
 * (user int, item int, rating fp32 = float32(float64(rating)/max_rating)). */
typedef struct {
  int32_t user;
  int32_t item;
  float rating;
  int32_t pad;
} ure_inter_t;

/* One shard model + its training data: the state Scratch.train builds
 * (method/scratch.py:59,65-69): MF tables (method/utils.py:30-43), SGD momentum
 * buffers, dense gradient scratch, and the shard's DataLoader contents. */
typedef struct {
  const ure_inter_t* inter; /* [n] the shard's training interactions                      */
  const int32_t* perm;      /* [n_epochs_total][n] explicit visiting orders, or NULL for   */
                            /* the keyed Feistel permutation (csrc/feistel.cuh)             */
  float* P;                 /* [n_user, d] user table                                      */
  float* Q;                 /* [n_item, d] item table                                      */
  float* bufP;              /* [n_user, d] momentum buffer (zero before the first step)    */
  float* bufQ;              /* [n_item, d]                                                 */
  float* gP;                /* [n_user, d] gradient scratch (zero on entry, zero on exit)  */
  float* gQ;                /* [n_item, d]                                                 */
  double* sse;              /* [n_epochs_total] per-epoch sum of squared errors (+=)       */
  int32_t* lastP;           /* lazy mode only: [n_user] steps applied to each row (bit 31: touched flag) */
  int32_t* lastQ;           /* lazy mode only: [n_item]                                    */
  int32_t* touched;         /* lazy mode only: [2][2][1 + batch] per step parity and table: count, row list */
  ure_inter_t* inter_u;     /* owner mode only: [n] records sorted by user, pad = index in `inter`          */
  ure_inter_t* inter_i;     /* owner mode only: [n] records sorted by item, pad = index in `inter`          */
  int32_t* off_u;           /* owner mode only: [n_user + 2] row offsets into inter_u (zero on entry of     */
                            /*    ure_mf_owner_prepare; entries 0..n_user valid afterwards)                 */
  int32_t* off_i;           /* owner mode only: [n_item + 2]                                                */
  int32_t* perm_inv;        /* owner mode with explicit `perm`: [n_epochs_total][n] inverse visiting orders */
  ure_inter_t* tmp_u;       /* owner mode only: [n] scratch of the radix sort                                */
  ure_inter_t* tmp_i;       /* owner mode only: [n] scratch of the radix sort                                */
  int32_t n;                /* interactions in the shard                                   */
  int32_t n_user;           /* rows of P                                                   */
  int32_t n_item;           /* rows of Q                                                   */
  int32_t shard_id;         /* Feistel key component                                       */
  uint32_t perm_seed;       /* Feistel key component                                       */
  int32_t group;            /* warp group (0 or 1) that trains this shard, see ure_mf_train        */
} ure_mf_shard_t;

typedef struct {
  int32_t d;            /* embedding dimension k (config.py:19): 8,16,32,64 or 128          */
  int32_t batch;        /* config.py:26                                                      */
  float lr0;            /* config.py:27                                                      */
  float lr_decay;       /* config.py:28, StepLR gamma (scratch.py:69)                        */
  int32_t lr_step;      /* StepLR step_size = 50 epochs (scratch.py:69)                      */
  float weight_decay;   /* config.py:20 lam                                                  */
  float momentum;       /* config.py:29                                                      */
  int32_t mode;         /* URE_MF_DENSE / URE_MF_LAZY / URE_MF_OWNER (below)                 */
  const float* decay;   /* lazy: DEVICE table [decay_len][4] of M^n = (a11,a12,a21,a22), the */
                        /*    n-step gradient-free update [w;buf] <- M^n [w;buf]; else NULL   */
  int32_t decay_len;    /* lazy: number of table entries (>= total steps + 1)                */
  int32_t owner_cap_rows;  /* OWNER: max owned rows of a CTA, from ure_mf_owner_prepare's plan      */
  int32_t owner_cap_slots; /* OWNER: max owned interactions of a CTA, rounded up to a multiple of 16 */
  int32_t owner_flags;     /* OWNER: bit 0 = keep the record cache in shared memory; bit 1 = the schedule
                            * pre-pass re-reads the record indices instead of caching them (large CTAs) */
  int32_t owner_spe_cap;   /* OWNER: max steps per epoch of a shard (plan)                           */
  int32_t owner_sched_rows;/* OWNER: epochs per shard the schedule tables hold                       */
  uint16_t* owner_sched;   /* OWNER: DEVICE [owner_sched_rows][owner_sched_stride] batch lists       */
  int32_t* owner_sched_off;/* OWNER: DEVICE [owner_sched_rows][#SMs][owner_spe_cap + 1] list offsets */
  int64_t owner_sched_step0;  /* OWNER: global step the schedule window starts at                    */
  int64_t owner_sched_stride; /* OWNER: slots of one schedule row = sum over the shards of 2 n       */
  int32_t owner_cap_list;  /* OWNER: batch-list entries a CTA stages in shared memory (multiple of 16, <=
                            * owner_cap_slots); a longer list is read from the schedule table directly  */
  int32_t owner_max_n;     /* OWNER: largest shard size n (sizes the round tables of the short-epoch schedule
                            * pre-pass); 0 = always use the general pre-pass                                */
  const struct ure_mf_runs_s* runs; /* RUNS: DEVICE table [n_shards] of the row slots / step lists (below)  */
  int32_t runs_rows;       /* RUNS: epochs per shard the step lists hold                                    */
  int32_t runs_spe_cap;    /* RUNS: max steps per epoch of a shard (< 1024)                                 */
  int64_t runs_step0;      /* RUNS: global step the list window starts at                                   */
  void* owner_plan;        /* OWNER: NULL, or the DEVICE workspace of ure_mf_train.  When set, ure_mf_owner_schedule checks
                            * ON THE DEVICE, CTA by CTA, that owner_cap_rows / owner_cap_slots / owner_spe_cap cover the
                            * plan, and leaves error code 2 in the workspace (int32 at byte 16) if they do not; ure_mf_train
                            * then trains nothing.  A caller may thus queue both launches with the capacities of an earlier
                            * plan of the same shapes instead of waiting for this plan's read-back (and skip the plan
                            * kernel: URE_BATCH_NO_PLAN), and repeats the pass with the exact plan when the code comes back */
} ure_mf_hparams_t;

/* RUNS schedule: per-shard state next to the ure_mf_shard_t entry, which still carries inter_u / inter_i of
 * ure_mf_owner_prepare and the public tables P / Q / bufP / bufQ that ure_mf_runs_init reads and
 * ure_mf_runs_flush writes). */
typedef struct ure_mf_runs_s {
  float* slotP;            /* [2][n_user][2 d]: two versions of every user row, each [w | momentum]        */
  float* slotQ;            /* [2][n_item][2 d]                                                             */
  unsigned long long* metaP; /* [n_user] version tag: steps applied to the previous version << 32 |         */
  unsigned long long* metaQ; /* [n_item]   steps applied to the current version << 1 | current slot         */
  uint32_t* list_u;        /* [runs_rows][n] slots of inter_u grouped by step, row order inside a step      */
  uint32_t* list_i;        /* [runs_rows][n] the same for inter_i                                           */
  int32_t* loff_u;         /* [runs_rows][runs_spe_cap + 1] first entry of every step's group               */
  int32_t* loff_i;
} ure_mf_runs_t;

/* ure_mf_hparams_t::mode -- three schedules of the SAME arithmetic (baseTrain + dense optim.SGD):
 *   DENSE  gradients scattered with L2 vector atomics (into the momentum arrays, pre-scaled), then a dense
 *          sweep; two grid barriers per step.  gP / gQ are not touched.
 *   LAZY   closed-form catch-up of untouched rows (M^n table) instead of the dense sweep.
 *   OWNER  owner-computes: every CTA owns a slice of user rows and a slice of item rows of ONE shard
 *          (weights + momentum resident in shared memory), walks its own interactions of the batch from
 *          the user-sorted and the item-sorted copy of the records, accumulates row gradients in
 *          registers (no atomics, no gradient arrays) and applies the SGD update in the same pass;
 *          weights are published double-buffered (P/Q and gP/gQ alternate) so one barrier per step
 *          among the shard's CTAs suffices.  Needs ure_mf_owner_prepare and n_shards <= #SMs. */
#define URE_MF_DENSE 0
#define URE_MF_LAZY 1
#define URE_MF_OWNER 2
#define URE_MF_RUNS 3     /* owner-computes for tables in HBM: sorted step lists, whole runs of a row per warp,
                           * two row versions + a tag instead of a second barrier (csrc/mf_train_runs.cu);
                           * needs ure_mf_owner_prepare (sorted copies), ure_mf_runs_init, ure_mf_runs_schedule
                           * and, before the public tables are read, ure_mf_runs_flush */

const char* ure_last_error(void);
int ure_abi_version(void);

/* Asynchronous copy of `bytes` from device memory to PAGE-LOCKED host memory on `stream` (results of a pass:
 * user_mat / item_mat tables, method/scratch.py:131-144 -- one call per contiguous run of tables). */
int ure_copy_to_host_async(void* h_dst, const void* d_src, int64_t bytes, void* stream);
/* ... and the other direction: page-locked host memory -> device (the float64 [3, n] arrays of read.py:64-68). */
int ure_copy_to_device_async(void* d_dst, const void* h_src, int64_t bytes, void* stream);

/* Bytes of device scratch ure_mf_train needs (grid barrier + step tables). */
int64_t ure_mf_train_workspace_bytes(void);

/* baseTrain (method/utils.py:46-111) for ALL shards of `d_shards` at once, for global steps
 * [step_begin, step_end).  Shard s runs batch (t mod spe_s) of its epoch (t div spe_s),
 * spe_s = ceil(n_s/batch), and is idle once it has done `epochs` epochs.  One persistent cooperative
 * launch, one 32-warp CTA per SM.  Shards are independent, so the warps of every CTA are split into two
 * groups: the first `warps_group0` warps train the shards with group == 0, the others those with
 * group == 1, each group with its own grid barrier, so one group's barrier latency is covered by the
 * other's work.  warps_group0 = 32 runs everything as one group (required when there is one shard).
 * Balance: warps_group0 / 32 ~ the share of the interactions that group 0's shards hold. */
int ure_mf_train(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp,
                 int epochs, int64_t step_begin, int64_t step_end, int warps_group0,
                 void* d_workspace, void* stream);

/* ---- BPR training (implicit feedback): the pairwise ranking objective over (user, rated item, unrated item) triples.
 * Per shard, the seen lists of ure_seen_lists built from the records the launch trains (never the whole file: a
 * negative excluded by data of a later SISA slice would make the slice checkpoints depend on it). */
typedef struct {
  const int64_t* seen_off;  /* [n_user + 1] row offsets into seen_items (user = the row in the shard's user table) */
  const int32_t* seen_items;/* the items of each user's training records, ascending                                */
} ure_bpr_shard_t;

/* ure_mf_train with the BPR objective, DENSE schedule only (hparams.mode = URE_MF_DENSE, else URE_EUNSUPPORTED);
 * d_bpr: DEVICE table [n_shards] of ure_bpr_shard_t.  Every record (u, i) is a positive (its rating is not used).
 * Epoch e's negative of record idx is the first of 16 candidates c_t = mulhi32(mix32(h + t * 0x85EBCA77), n_item),
 * h = mix32(key ^ (idx * 0x9E3779B1 + 0x7F4A7C15)), key = perm_key(perm_seed, shard_id, e) (csrc/feistel.cuh), that
 * is not in u's seen list; if all 16 are seen the triple is dropped.  With x = P[u].(Q[i] - Q[j]), c = sigmoid(-x):
 * loss softplus(-x), gradients -c (Q[i] - Q[j]) for P[u], -c P[u] for Q[i], +c P[u] for Q[j], PRE-step weights;
 * then the same dense SGD (momentum, L2, StepLR).  sse[e] += the sum of softplus(-x) over the epoch's triples. */
int ure_mf_train_bpr(const ure_mf_shard_t* d_shards, const ure_bpr_shard_t* d_bpr, int n_shards,
                     const ure_mf_hparams_t* h_hp, int epochs, int64_t step_begin, int64_t step_end, int warps_group0,
                     void* d_workspace, void* stream);

/* Diagnostics and tests: d_neg[idx] = the negative of record idx of one shard in epoch `epoch` (-1: dropped), as
 * ure_mf_train_bpr draws it.  d_tries (may be NULL): the number of candidates drawn for each record. */
int ure_bpr_negatives(const ure_inter_t* d_inter, int32_t n, int32_t n_item, const int64_t* d_seen_off,
                      const int32_t* d_seen_items, uint32_t perm_seed, int32_t shard_id, int32_t epoch, int32_t* d_neg,
                      int32_t* d_tries, void* stream);

/* Owner mode set-up, once per shard table (asynchronous, no host sync): builds inter_u / inter_i /
 * off_u / off_i (row histogram + scan; STABLE radix sort of the records by user and by item, so the whole
 * training is reproducible bit for bit) and perm_inv for shards with an explicit perm, then plans the CTA ownership and writes into the first 16 bytes of d_workspace
 * int32 {max owned rows of a CTA, max owned interactions of a CTA, max steps per epoch of a shard,
 * dynamic shared-memory bytes available}: the caller reads them back once, fills hparams.owner_cap_rows /
 * owner_cap_slots / owner_cap_list / owner_spe_cap / owner_flags, allocates the schedule tables, and must not start mode OWNER
 * when ure_mf_owner_smem_bytes exceeds what is available (ure_mf_train refuses it loudly as well). */
int64_t ure_mf_owner_radix_bytes(int n_shards);     /* size of d_radix_hist below */
int ure_mf_owner_prepare(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp,
                         int epochs, int max_rows /* largest n_user / n_item of a shard */,
                         int32_t* d_radix_hist, void* d_workspace, void* stream);

/* Dynamic shared memory per CTA the OWNER schedule needs for these capacities (training kernel and
 * schedule pre-pass, whichever is larger).  flags as hparams.owner_flags; cap_list as hparams.owner_cap_list: with
 * bit 0 (record cache) it must equal cap_slots, without it 10 bytes are needed per staged list entry, so a caller
 * short of shared memory lowers cap_list (batch lists longer than it are read from the schedule table). */
int64_t ure_mf_owner_smem_bytes(int d, int cap_rows, int cap_slots, int cap_list, int spe_cap, int flags);

/* OWNER mode, before ure_mf_train: fill the schedule tables for the window of owner_sched_rows epochs per
 * shard that starts at global step `step0` (epoch step0 / spe_s of shard s): for every training CTA, epoch
 * and step, the sorted list of the CTA's interactions in that step's batch -- the inverse of the epoch's
 * visiting order (keyed Feistel permutation or perm_inv), evaluated in one embarrassingly parallel pass.
 * ure_mf_train may then run any steps [a, b) with step0 <= a whose epochs lie inside the window
 * (hparams.owner_sched_step0 = step0); a step outside it stops the shard and raises the workspace's error
 * word (int32 at byte 16). */
int ure_mf_owner_schedule(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp,
                          int epochs, int64_t step0, void* stream);

/* ---- Native host runtime of a K-shard training batch (replaces the per-shard Python bookkeeping of the K
 * sequential Scratch.train set-ups, method/sisa.py:33-36, 86-89 -> scratch.py:59-69) ------------------------------
 * One device allocation of the caller (the "arena") holds everything the batch needs; the library lays it out,
 * writes the descriptor table, clears what must start at zero and queues the owner set-up; nothing is allocated by
 * the library and nothing synchronises. */
typedef struct {
  const ure_inter_t* inter; /* DEVICE records of the shard; the user field is the row in the shard's user table   */
  const int32_t* perm;      /* DEVICE explicit visiting orders [epochs][n], or NULL (keyed Feistel permutation)    */
  int32_t n;                /* interactions                                                                        */
  int32_t n_user;           /* rows of the shard's user table                                                      */
  int32_t shard_id;         /* Feistel key component (model id, method/sisa.py:35)                                 */
  int32_t group;            /* warp group of the DENSE schedule (ure_mf_train)                                     */
} ure_mf_batch_shard_t;

typedef struct {            /* byte offsets into the arena (multiples of 256) and the numbers they were sized from */
  int64_t total;            /* bytes the caller allocates                                                          */
  int64_t table;            /* ure_mf_shard_t [K]: the descriptor table ure_mf_train / ure_mf_owner_* take         */
  int64_t ws;               /* ure_mf_train_workspace_bytes()                                                      */
  int64_t W;                /* fp32 [rows_total + K*n_item, d]: user tables of shard 0..K-1, then the K item tables */
                            /* -- the CALLER fills it (N(0,1) init, method/utils.py:38-40) before ure_mf_train     */
  int64_t Z;                /* fp32 [2][rows_total + K*n_item, d]: momentum, gradient scratch (zeroed by setup)    */
  int64_t sse;              /* fp64 [K][max(1, epochs)] (zeroed by setup)                                          */
  int64_t zero_end;         /* end of the region setup clears                                                     */
  int64_t rec, off, radix, perm_inv, sched, sched_off;   /* owner schedule only                                   */
  int64_t rows_total, n_total, sched_stride;
  int32_t spe_cap, max_rows, max_n, grid, owner, sched_rows;
} ure_mf_batch_layout_t;

/* Layout for these shards.  owner != 0 asks for the OWNER schedule's buffers when the weights + momentum of all rows
 * can fit the SMs' shared memory (out->owner tells); sched_bytes_cap bounds the schedule tables (>= 2 epochs). */
int ure_mf_batch_layout(const ure_mf_batch_shard_t* h_shards, int n_shards, int n_item, int d, int batch,
                        int epochs, int owner, int64_t sched_bytes_cap, ure_mf_batch_layout_t* out);

/* Descriptor table -> arena (through h_stage: page-locked host memory of the caller, >= 176*K + 64 bytes, not to be
 * reused before the stream has passed this call), clears momentum / gradient scratch / losses / workspace / row
 * offsets, queues ure_mf_owner_prepare when lay->owner, and queues the copy of the plan (4 int32, see
 * ure_mf_owner_prepare) to h_stage + 176*K.  The weights (lay->W) are left to the caller. */
#define URE_BATCH_NO_PLAN 1       /* flags: do not compute / copy the plan (the launch runs on remembered capacities,
                                   * hparams.owner_plan set) */
int ure_mf_batch_setup(const ure_mf_batch_shard_t* h_shards, int n_shards, int n_item, const ure_mf_hparams_t* h_hp,
                       int epochs, uint32_t perm_seed, void* d_arena, const ure_mf_batch_layout_t* lay, void* h_stage,
                       int flags, void* stream);

/* After the stream has passed ure_mf_batch_setup: turn the plan into launch parameters (hp->mode = OWNER, owner_*
 * capacities, the shared-memory configuration -- record cache first, then staged lists -- and the schedule-table
 * pointers inside the arena).  Returns 1 when the OWNER schedule can run, 0 when the caller must use DENSE with the
 * same descriptor table, < 0 on error.  force_flags >= 0 pins the configuration (tests).  h_info (may be NULL):
 * int32 [8] = {fits, flags, cap_list, cap_rows, cap_slots, spe_cap, smem needed, smem available}. */
int ure_mf_batch_plan(const int32_t* h_plan, int n_shards, ure_mf_hparams_t* hp, void* d_arena,
                      const ure_mf_batch_layout_t* lay, int allow_cache, int force_flags, int force_list,
                      int32_t* h_info);

/* ---- RUNS schedule (mode URE_MF_RUNS) ---------------------------------------------------------------------------
 * ure_mf_runs_init: slot 0 of every row <- [P | bufP] / [Q | bufQ], tags cleared (once, before the first step).
 * ure_mf_runs_schedule: the step lists for the window of runs_rows epochs per shard that starts at global step
 *   `step0` -- a stable counting sort of the user-sorted / item-sorted slots by the step whose batch holds them (the
 *   inverse of the epoch's visiting order).  d_scratch: ure_mf_runs_scratch_bytes(n_shards, max_n, rows, spe_cap).
 * ure_mf_train with mode RUNS then runs any steps of that window (hparams.runs_step0 = step0).
 * ure_mf_runs_flush: every row advanced to the current step and written to the public tables. */
int64_t ure_mf_runs_scratch_bytes(int n_shards, int64_t max_n, int rows, int spe_cap);
int ure_mf_runs_init(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp, void* stream);
int ure_mf_runs_schedule(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp, int epochs,
                         int64_t step0, int64_t max_n, void* d_scratch, void* stream);
int ure_mf_runs_flush(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp, int epochs,
                      int64_t step_now, void* stream);

/* Diagnostics (tracing): record six SM-clock stamps per CTA and step -- step start, tables ready,
 * gradients issued, barrier 1 passed, sweep issued, barrier 2 passed -- for the first `steps` steps of
 * the following ure_mf_train calls into d_trace [steps][ure_mf_grid_size()][6] int64; NULL = off. */
int ure_mf_train_trace(void* d_workspace, int64_t* d_trace, int steps, void* stream);
int ure_mf_grid_size(void);
/* Diagnostics: bit 0 skips the gradient scatter, bit 1 uses the identity visiting order, bits 8..13 force
 * warps_group0 (timing experiments only). */
int ure_mf_debug_flags(void* d_workspace, unsigned flags, void* stream);

/* Lazy mode: bring every row of every shard up to date (before the tables are read by anything else):
 * rows whose step count is below the shard's own (min(step_now, spe_s*epochs)) are advanced with M^n.
 * h_shards is the HOST copy of the descriptor table.  No-op in dense mode. */
int ure_mf_flush(const ure_mf_shard_t* h_shards, int n_shards, const ure_mf_hparams_t* h_hp,
                 int epochs, int64_t step_now, void* stream);

/* Ensemble score of baseTest (method/utils.py:141-148):
 * score[j] = (sum_k P_k[u_j].Q_k[i_j]) / denom;  *sse += sum_j (score[j]-r_j)^2.
 * denom = K gives torch.stack(preds).mean(0); denom = 1 gives the partial sum a rank
 * contributes before the cross-GPU all-reduce (then ure_score_finalize).
 * d_P / d_Q are device arrays of K table pointers.  d_score and d_sse may be NULL. */
int ure_ensemble_score(const float* const* d_P, const float* const* d_Q, int n_models, int d,
                       const ure_inter_t* d_inter, int64_t n, float denom, float* d_score,
                       double* d_sse, void* stream);

/* score[j] = sum[j] / denom (in place allowed); *sse += sum_j (score[j]-r_j)^2. */
int ure_score_finalize(const float* d_sum, const ure_inter_t* d_inter, int64_t n, float denom,
                       float* d_score, double* d_sse, void* stream);

/* HR@10 / NDCG@10 of baseTest (method/utils.py:166-184) over user segments.
 * Segment s covers rows d_order[d_seg[s] .. d_seg[s+1]) (d_order NULL = identity).
 * d_out[0] += sum_u ndcg_u ; d_out[1] += sum_u hr_u ; d_out[2] += #users.
 * Tie rule: descending value, later index first (np.argsort(kind='stable')[::-1]), in NumPy's order
 * of floats: a NaN score ranks above +inf and ties with every other NaN; -0 and +0 tie. */
int ure_rank_metrics(const ure_inter_t* d_inter, const float* d_score, const int32_t* d_order,
                     const int64_t* d_seg, int64_t n_seg, double* d_out, void* stream);

/* Many evaluations in ONE pair of launches (grid.y = job): the per-epoch in-training evaluations of
 * method/scratch.py:83-97 (two baseTest calls per shard and epoch).  Every job is what ure_ensemble_score +
 * ure_rank_metrics do for one (model list, test set): out[0] += sum of squared errors, out[1..3] += (sum NDCG@10,
 * sum HR@10, users).  score: n floats of scratch per job.  max_n / max_seg: the largest n / n_seg of the jobs. */
typedef struct {
  const float* const* P;   /* DEVICE table of n_models user-table pointers                                   */
  const float* const* Q;   /* DEVICE table of n_models item-table pointers                                   */
  const ure_inter_t* inter;
  const int32_t* order;    /* as ure_rank_metrics (or NULL)                                                  */
  const int64_t* seg;      /* [n_seg + 1]                                                                    */
  float* score;            /* [n] scratch                                                                    */
  double* out;             /* [4], zero on entry                                                             */
  int64_t n, n_seg;
  int32_t n_models;
  float denom;             /* usually n_models                                                               */
} ure_eval_job_t;
int ure_eval_jobs(const ure_eval_job_t* d_jobs, int n_jobs, int d, int64_t max_n, int64_t max_seg, void* stream);

/* Data ingest (what RatingData.__init__ + __getitem__ do on the host, read.py:111-113,118-124): the float64
 * [3, n] array readRating hands over (rows: user id, item id, rating / max_rating; row stride ld elements),
 * already on the device, becomes packed records: user = int(u) -- or d_row_of[int(u)], the row inside a
 * compact per-shard user table, when d_row_of != NULL -- item = int(i), rating = float32(r). */
int ure_pack_interactions_f64(const double* d_cols, int64_t n, int64_t ld, const int32_t* d_row_of,
                              int32_t n_map, ure_inter_t* d_out, void* stream);

/* readRating's row filter and shard split (read.py:36-68) on the device: ONE stable partition of the whole ratings
 * table by shard.  d_cols: the float64 table as read from the CSV, field c of rating j at d_cols[j*rs + c*cs] (c = uid, iid,
 * rating; [n][3] row-major: rs=3, cs=1; [3][n]: rs=1, cs=n); d_owner[u]:
 * shard of user u (-1: none), d_deleted[u] != 0: user u is deleted (NULL: nobody).  d_out [n]: every shard's
 * records (user id, item id, float32(rating / max_rating)) as one contiguous run in file order;
 * d_shard_off int64 [n_shards + 1]: the runs' starts, d_shard_off[n_shards] = rows kept.
 * d_hist: int32 scratch [ure_partition_blocks()][256].  n_shards <= 254. */
int ure_partition_blocks(void);
int ure_partition_interactions(const double* d_cols, int64_t n, int64_t rs, int64_t cs, double max_rating,
                               const int32_t* d_owner, const uint8_t* d_deleted, int32_t n_map, int n_shards,
                               ure_inter_t* d_out, int32_t* d_hist, int64_t* d_shard_off, void* stream);
/* ure_partition_interactions that also drops deleted ratings (interaction-level unlearning): a row of user u whose
 * item int(i) lies in d_del_item[d_del_off[u] .. d_del_off[u+1]) goes with the dropped rows.  d_del_off: int64
 * [n_map + 1], d_del_item: int32, ascending within each user (duplicates allowed) -- the layout ure_seen_lists builds
 * from the deleted (user, item) pairs.  Both NULL: exactly ure_partition_interactions. */
int ure_partition_interactions_del(const double* d_cols, int64_t n, int64_t rs, int64_t cs, double max_rating,
                                   const int32_t* d_owner, const uint8_t* d_deleted, int32_t n_map, int n_shards,
                                   const int64_t* d_del_off, const int32_t* d_del_item, ure_inter_t* d_out,
                                   int32_t* d_hist, int64_t* d_shard_off, void* stream);
/* out[j] = in[j] with user -> d_row_of[user] (the row inside a compact per-shard user table). */
int ure_remap_users(const ure_inter_t* d_in, int64_t n, const int32_t* d_row_of, int32_t n_map,
                    ure_inter_t* d_out, void* stream);

/* HOST helper of the ingest path: copy `bytes` from pageable memory into a (pinned) staging buffer with
 * non-temporal stores, so that the DMA engine reads DRAM and not other cores' caches.  Thread-safe on disjoint
 * ranges (the caller's thread pool splits the arrays); dst 16-byte aligned. */
int ure_host_stage_copy(void* h_dst, const void* h_src, int64_t bytes);

/* Per-user segments of a test set (the host dict of method/utils.py:151-161): a STABLE sort of the records by user
 * id (a user's rows stay in file order, which the ranking's tie rule depends on), d_order[x] = index of the x-th row
 * in that order, d_seg[u] .. d_seg[u+1] = the rows of user u (int64 [n_user + 1]; users without rows give empty
 * segments, which ure_rank_metrics skips).  d_scratch: ure_user_segments_scratch_bytes(n, n_user) bytes. */
int64_t ure_user_segments_scratch_bytes(int64_t n, int n_user);
int ure_user_segments(const ure_inter_t* d_inter, int64_t n, int n_user, int32_t* d_order, int64_t* d_seg,
                      void* d_scratch, void* stream);

/* ---- Top-N recommendation over the whole catalogue (no counterpart in the reference, whose baseTest ranks each
 * user's test items only).  score(u, i) = scale * sum_t P[u,t] * S[i,t] in fp32, S = sum_k Q_k, scale = 1/K. */

/* Seen lists: d_off int64 [n_user + 1], d_items int32 [n]: the items of user u's records in ascending order at
 * d_items[d_off[u] .. d_off[u+1]) (a stable radix sort by item, then by user; no host pass).  User and item ids must lie
 * in [0, n_user) and [0, n_item); the library does not check them (that would need a synchronisation): the Python
 * wrapper kernels.seen_lists does.  d_scratch: ure_seen_lists_scratch_bytes(n, n_user) bytes. */
int64_t ure_seen_lists_scratch_bytes(int64_t n, int n_user);
int ure_seen_lists(const ure_inter_t* d_inter, int64_t n, int n_user, int n_item, int64_t* d_off, int32_t* d_items,
                   void* d_scratch, void* stream);

/* d_S [n_item, d] = sum over k < n_models of d_Q[k] (a device array of table addresses), summed in k order.
 * d a multiple of 4. */
int ure_item_sum(const float* const* d_Q, int n_models, int64_t n_item, int d, float* d_S, void* stream);

/* d_lo[j] = d_X[j] - trunc_tf32(d_X[j]) for j < n (n a multiple of 4): the lo operand of the 3-term tf32 split. */
int ure_split_lo(const float* d_X, int64_t n, float* d_lo, void* stream);

/* Per requested user d_users[r] (r < m; any order, duplicates allowed), the top_n items by score, descending, ties to
 * the smaller item id, never an item of the user's seen list (d_seen_off / d_seen from ure_seen_lists, or both NULL:
 * nothing excluded).  d_items int32 [m, top_n], d_scores fp32 [m, top_n]; a list with fewer eligible items than top_n
 * is padded with item -1 and score -inf, as is the row of an id outside [0, n_user).  d_S_lo: ure_split_lo of d_S.
 * tcgen05 kind::tf32 with the 3-term hi/lo split (fp32-accurate); the top-N is kept in the epilogue, the score matrix
 * is never written.  d in {8,16,32,64,128}, 1 <= top_n <= 64 (else URE_EUNSUPPORTED), scale > 0.
 * d_scratch: ure_topn_scratch_bytes(m, n_item, d, top_n) bytes (0: may be NULL). */
int64_t ure_topn_scratch_bytes(int64_t m, int64_t n_item, int d, int top_n);
int ure_topn(const float* d_P, int n_user, const float* d_S, const float* d_S_lo, int64_t n_item, int d,
             const int32_t* d_users, int64_t m, const int64_t* d_seen_off, const int32_t* d_seen, int top_n, float scale,
             int32_t* d_items, float* d_scores, void* d_scratch, void* stream);

/* Full-catalogue metrics of top-N lists (d_items [m, top_n] for d_users [m]) against test records grouped by
 * ure_user_segments (d_order may be NULL when the records are already grouped; d_seg int64 [n_user + 1]).  rel(u) =
 * the user's distinct test items with rating >= 4/5 (method/utils.py:175,180); rows whose user has none are skipped.
 * d_out fp64 [4] += (sum HR@N, sum Recall@N = hits/|rel|, sum NDCG@N, rows counted), with
 * NDCG@N = sum_{p < N, hit} 1/log2(p+2) / sum_{p < min(N, |rel|)} 1/log2(p+2).  top_n <= 64 (else URE_EUNSUPPORTED). */
int ure_topn_metrics(const int32_t* d_items, const int32_t* d_users, int64_t m, int top_n, const ure_inter_t* d_test,
                     const int32_t* d_order, const int64_t* d_seg, int n_user, double* d_out, void* stream);

/* ---- Learned combination of the shard models (UltraRE's combination estimator; the reference scores with the plain
 * mean).  Per owner group g: s(u, i) = b_g + sum_k w_gk x_k with x_k = P[u].Q_k[i] (P the merged user table)
 * = b_g + P[u].T_g[i], T_g = sum_k w_gk Q_k.  The ridge solve of (w_g, b_g) is (K+1) x (K+1) and runs on the host. */
#define URE_COMBINE_MAX_MODELS 64
#define URE_COMBINE_GRAM_CTAS 128   /* CTAs per group of ure_combine_gram: fixed, so the summation order is too */

/* Gram of the features over the records of n_groups groups (d_inter / d_n: device arrays of n_groups record
 * pointers and row counts), K = n_models item tables d_Q (device array of pointers), P [*, d].  Per group g,
 * d_out[g * E ..] with E = (K+1)(K+2)/2 + (K+1) + 1, fp64: the upper triangle of sum [x;1][x;1]^T row by row, then
 * sum [x;1] * r, then the row count.  x_k = sum_t P[u,t] * Q_k[i,t] with the fp32 entries multiplied and summed in
 * fp64; the sums are fp64 without atomics, folded in a fixed order: two calls give the same bits.  d_scratch: n_groups *
 * URE_COMBINE_GRAM_CTAS * E doubles.  Ids are not checked.  K > URE_COMBINE_MAX_MODELS or d not in
 * {8,16,32,64,128}: URE_EUNSUPPORTED. */
int ure_combine_gram(const float* d_P, const float* const* d_Q, int n_models, int d, const ure_inter_t* const* d_inter,
                     const int64_t* d_n, int n_groups, double* d_out, double* d_scratch, void* stream);

/* d_T [n_out, n_item, d]: T_o = sum_k d_w[o * n_models + k] * d_Q[k] in k order (t = w_0 q_0, then fma), fp32
 * weights; the weighted sibling of ure_item_sum.  d a multiple of 4. */
int ure_item_wsum(const float* const* d_Q, int n_models, const float* d_w, int n_out, int64_t n_item, int d,
                  float* d_T, void* stream);

/* score[j] = d_b[s] + P[u_j].T_s[i_j] with s = d_owner[u_j], or the last slot n_slots - 1 (the mean combination) when
 * d_owner[u_j] < 0; d_T [n_slots, n_item, d], d_b fp32 [n_slots].  *d_sse += sum_j (score[j] - r_j)^2 as
 * ure_ensemble_score (d_score and d_sse may be NULL).  Ids and owner values are not checked. */
int ure_group_score(const float* d_P, const float* d_T, int n_slots, int64_t n_item, int d, const float* d_b,
                    const int32_t* d_owner, const ure_inter_t* d_inter, int64_t n, float* d_score, double* d_sse,
                    void* stream);

/* Affected-shard routing (method/sisa.py:76-81): flags[owner[u]] = 1 for u in del. */
int ure_route_deletions(const int32_t* d_owner, int32_t n_user, const int32_t* d_del, int32_t n_del,
                        int32_t* d_flags, int32_t n_shards, void* stream);

/* Merge of owner rows (method/sisa.py:52-58 learn, 107-113 unlearn):
 * row u of d_merged <- P_{owner[u]}[row_of[u]] when owner[u] >= 0 and
 * (d_retrain == NULL or d_retrain[owner[u]] != 0); rows with owner[u] < 0 are
 * zeroed when zero_unowned != 0 (learn), else left as they are (unlearn).
 * d_row_of NULL = the shard table is indexed by global user id. */
int ure_merge_user_rows(const float* const* d_P, const int32_t* d_owner, const int32_t* d_row_of,
                        const int32_t* d_retrain, float* d_merged, int32_t n_user, int d,
                        int zero_unowned, void* stream);

/* Squared-euclidean cost matrix of ot_cluster (method/utils.py:637), transposed to
 * [n, kpad] row major: M[i,j] = ||x_i||^2 + ||c_j||^2 - 2 x_i.c_j, the contraction on
 * tcgen05 (kind::tf32, 3-term hi/lo split = fp32-accurate).  Columns j >= k are
 * filled with +inf.  d multiple of 8, d <= 128; kpad = 8 or a multiple of 16, <= 256.
 * d_inertia (may be NULL): += sum_i min_j M[i,j] (utils.py:638). */
int ure_cost_matrix(const float* d_X, int64_t n, int d, const float* d_C, int k, int kpad,
                    float* d_M, double* d_inertia, void* stream);

/* Same contraction on CUDA cores (fp32 FMA): the check for the tcgen05 kernel. */
int ure_cost_matrix_simt(const float* d_X, int64_t n, int d, const float* d_C, int k, int kpad,
                         float* d_M, double* d_inertia, void* stream);

/* One Sinkhorn column pass (replaces the ot.emd call, utils.py:641-644):
 * for every row i: P_ij = a_i * softmax_j((g_j - M_ij)/eps);  d_colsum[j] += sum_i P_ij.
 * a_i = 1/n_total.  d_colsum is double [kpad], zero on entry.  The sums are accumulated in the log domain
 * (per-column reference exponents): a column whose entries all lie hundreds of binades below their row maxima
 * still gets its exact, non-zero sum (down to 2^-960), so no potential can run away after a stale warm start. */
int ure_sinkhorn_colsum(const float* d_M, int64_t n, int k, int kpad, const float* d_g, float eps,
                        double n_total, double* d_colsum, void* stream);

/* g_j += eps * (log(1/k) - log(colsum_j)); re-zeroes d_colsum. */
int ure_sinkhorn_update_g(float* d_g, double* d_colsum, int k, float eps, void* stream);

/* Whole single-GPU Sinkhorn: h_eps[s], h_iters[s] for s < n_stages (epsilon scaling), starting from the
 * potentials in d_g (zeros = cold start).  Small problems (a CTA's rows of M fit in shared memory) run as ONE
 * persistent cooperative launch with a grid barrier per iteration and, when tol > 0, leave a stage early once
 * max_j |colsum_j - 1/k| * k < tol; large problems run the split-phase kernels for every scheduled iteration.
 * d_workspace: ure_sinkhorn_workspace_bytes() bytes. */
int64_t ure_sinkhorn_workspace_bytes(void);
int ure_sinkhorn(const float* d_M, int64_t n, int k, int kpad, float* d_g, const float* h_eps,
                 const int32_t* h_iters, int n_stages, float tol, void* d_workspace, void* stream);

/* Multi-GPU Sinkhorn in ONE persistent launch per GPU (SURVEY.md §8e, H6): the users (rows of d_M) are sharded
 * over `world` GPUs of one NVLink / NVSwitch domain; per iteration every GPU makes its column pass, stores its k
 * column sums into every peer's exchange buffer (peer-mapped symmetric memory) and raises a flag there; every GPU adds
 * the per-GPU sums in rank order (bit-identical potentials everywhere) -- no NCCL call, no launch between iterations.
 * h_xchg_ptrs: HOST array [world] of the device addresses of every rank's exchange buffer as mapped in THIS process
 * (own buffer included), each ure_sinkhorn_peer_xchg_bytes() bytes, zero-filled once when allocated and never reset.
 * call_base: a counter that is equal on all ranks and grows by more than the call's total iteration count from call
 * to call (flags carry call_base + iteration).  All ranks must make the same calls in the same order.  After the
 * call the int64 iters_done of the workspace is -1 if a peer did not arrive within a few seconds.
 * d_workspace: ure_sinkhorn_workspace_bytes() bytes. */
int64_t ure_sinkhorn_peer_xchg_bytes(void);
int ure_sinkhorn_peer(const float* d_M, int64_t n_local, double n_total, int k, int kpad, float* d_g,
                      const float* h_eps, const int32_t* h_iters, int n_stages, float tol,
                      const uint64_t* h_xchg_ptrs, int rank, int world, uint64_t call_base,
                      void* d_workspace, void* stream);

/* Row-normalised plan for given g: P[i,j] = (1/n_total) softmax_j((g_j - M_ij)/eps), [n,k] fp32. */
int ure_sinkhorn_plan(const float* d_M, int64_t n, int k, int kpad, const float* d_g, float eps,
                      double n_total, float* d_plan, void* stream);

/* label_i = argmax_j plan[i,j], first maximum wins (utils.py:647). plan fp64 or fp32, ld = row stride. */
int ure_assign_plan_f64(const double* d_plan, int64_t n, int k, int64_t ld, int32_t* d_label, void* stream);
int ure_assign_plan_f32(const float* d_plan, int64_t n, int k, int64_t ld, int32_t* d_label, void* stream);

/* label_i = argmax_j (g_j - M_ij) (== argmax of the Sinkhorn plan row), and the
 * centroid accumulators of utils.py:648: d_sum[j,:] += x_i, d_cnt[j] += 1 (double / int64). */
int ure_assign_centroids(const float* d_M, int64_t n, int k, int kpad, const float* d_g,
                         const float* d_X, int d, int32_t* d_label, double* d_sum, int64_t* d_cnt,
                         void* stream);

/* Centroid accumulators of utils.py:648 for GIVEN labels (after ure_balance_labels):
 * d_sum[j,:] += x_i, d_cnt[j] += 1 for j = d_label[i]. */
int ure_centroid_sums(const float* d_X, int64_t n, int d, const int32_t* d_label, int k, double* d_sum,
                      int64_t* d_cnt, void* stream);

/* Balanced rounding of the assignment (SURVEY.md H1 iv; the reference's exact EMD plan, utils.py:641-647, puts
 * exactly n/k users in every group): d_label / d_cnt = the argmax assignment of ure_assign_centroids and its group
 * sizes on entry; users are moved from over-full to under-full groups along successive shortest augmenting paths
 * of the group graph (edge j->l = the cheapest M_il - M_ij over the members of j), which keeps the assignment
 * cost-optimal for its sizes and ends at the minimum-cost assignment with floor(n/k)..ceil(n/k) users per group.
 * At most max_aug augmentations (one pass over M each).  d_workspace: ure_balance_workspace_bytes(k) bytes; after
 * the call its int32 words [32..34] hold {augmentations applied, users still to move, gave-up flag}.  k <= 128. */
int64_t ure_balance_workspace_bytes(int k);
int ure_balance_labels(const float* d_M, int64_t n, int k, int kpad, int32_t* d_label, int64_t* d_cnt,
                       int max_aug, void* d_workspace, void* stream);

/* ---- 'rating-ot' grouping: the points are the users' sparse rating rows (reference group.py, readSparseMat) ---- */
#define URE_SPARSE_OT_MAX_K 128   /* centroids of the sparse kernels: the balanced rounding's limit */

/* The cost matrix of ure_cost_matrix -- [n, kpad] row major, columns j >= k +inf, d_inertia (may be NULL)
 * += sum_i max(min_j M[i,j], 0) -- for sparse rows: M[i,j] = ||x_i||^2 - 2 x_i.c_j + ||c_j||^2.
 * x_i: the ratings of user i in CSR, entries d_off[i] .. d_off[i+1] (int64 [n + 1]) of d_item (int32, ascending within
 * a row; adjacent duplicates stand for their fp32 sum, the entry of SciPy's summed row) and d_val (fp32).
 * d_Ct: the centroids item-major, fp32 [n_item, kpad], columns j >= k zero; d_cnorm: fp64 [k] = ||c_j||^2.  The dot
 * products and ||x_i||^2 multiply fp32 values and add them in fp64; each cost is rounded to fp32 once.  The inertia is
 * added in a fixed order (the same bits on every call).  1 <= k <= URE_SPARSE_OT_MAX_K and kpad = the smallest of
 * 8, 16, .., 128 that holds k (else URE_EUNSUPPORTED).  d_scratch: ure_sparse_cost_scratch_bytes(n) bytes (only read
 * with d_inertia).  Item ids are not checked. */
int64_t ure_sparse_cost_scratch_bytes(int64_t n);
int ure_sparse_cost(const int64_t* d_off, const int32_t* d_item, const float* d_val, int64_t n, const float* d_Ct,
                    const double* d_cnorm, int k, int kpad, float* d_M, double* d_inertia, void* d_scratch,
                    void* stream);

/* Centroid sums of the sparse rows for given labels: the ratings in CSC, entries d_off[t] .. d_off[t+1] (int64
 * [n_item + 1]) of d_user (int32, ascending within a column; the fp32 sum of adjacent duplicates is the entry, as in
 * ure_sparse_cost) and d_val (fp32) for item t.  d_sum fp64 [n_item, kpad] = per item the sum of its
 * ratings by label d_label[user] (every entry written, 0 where there is none), each added in the column's order without
 * floating-point atomics: two calls give the same bits.  d_cnt int64 [k] = the users per label (set, not added).
 * k, kpad as ure_sparse_cost.  User ids and labels are not checked (a label outside [0, k) is neither summed nor
 * counted). */
int ure_sparse_centroid_sums(const int64_t* d_off, const int32_t* d_user, const float* d_val, int64_t n_item,
                             const int32_t* d_label, int64_t n_user, int k, int kpad, double* d_sum, int64_t* d_cnt,
                             void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ULTRARE_B200_H */
