// Deterministic negative sampler of the BPR training objective (ure_mf_train_bpr, ure_bpr_negatives).
//
// Record idx of a shard (user row u, item i) trains the triple (u, i, j) in epoch e.  Its negative j is the first
// of T = 16 candidates that is not in u's seen list (the items of u's records among the records the launch trains):
//   h   = mix32(key ^ (idx * 0x9E3779B1 + 0x7F4A7C15)),   key = perm_key(perm_seed, shard_id, e)  (feistel.cuh)
//   c_t = mulhi32(mix32(h + t * 0x85EBCA77), n_item)      t = 0 .. T-1, uniform in [0, n_item)
// all in uint32 arithmetic.  If all T candidates are seen the triple is dropped (j = -1: no loss, no gradient).
// The key is the epoch's visiting-order key, but the hash takes the record index, not its position in the
// visiting order, so a record's candidates do not depend on the permutation (explicit or Feistel).
// oracle/bpr.py restates this bit for bit.
#pragma once
#include <stdint.h>

#include "feistel.cuh"

namespace ure {

constexpr int kBprCandidates = 16;

__host__ __device__ __forceinline__ uint32_t bpr_record_hash(uint32_t key, uint32_t idx) {
  return mix32(key ^ (idx * 0x9E3779B1u + 0x7F4A7C15u));
}

__host__ __device__ __forceinline__ uint32_t bpr_candidate(uint32_t h, int t, uint32_t n_item) {
  return mulhi32(mix32(h + (uint32_t)t * 0x85EBCA77u), n_item);
}

// The negative of record idx (or -1), given u's seen list seen[lo, hi) (ascending; duplicates allowed): one binary
// search per candidate.  *tries (may be NULL) receives the number of candidates drawn.
__device__ __forceinline__ int bpr_negative(uint32_t key, uint32_t idx, const int32_t* __restrict__ seen, long long lo,
                                            long long hi, uint32_t n_item, int* tries = nullptr) {
  const uint32_t h = bpr_record_hash(key, idx);
  for (int t = 0; t < kBprCandidates; ++t) {
    const int c = (int)bpr_candidate(h, t, n_item);
    long long a = lo, b = hi;           // first position with seen[pos] >= c
    while (a < b) {
      const long long m = (a + b) >> 1;
      if (__ldg(seen + m) < c) a = m + 1; else b = m;
    }
    if (a == hi || __ldg(seen + a) != c) {
      if (tries) *tries = t + 1;
      return c;
    }
  }
  if (tries) *tries = kBprCandidates;
  return -1;
}

}  // namespace ure
