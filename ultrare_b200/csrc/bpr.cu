// BPR training (ure_mf_train_bpr: the DENSE schedule of mf_dense.cuh with the pairwise ranking objective) and
// ure_bpr_negatives, the sampler of bpr_sampler.cuh for every record of one shard and epoch.
#include "mf_dense.cuh"

namespace ure {
namespace {

__global__ void bpr_negatives_kernel(const ure_inter_t* __restrict__ inter, int n, uint32_t n_item,
                                     const int64_t* __restrict__ seen_off, const int32_t* __restrict__ seen,
                                     uint32_t key, int32_t* __restrict__ neg, int32_t* __restrict__ tries) {
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += gridDim.x * blockDim.x) {
    const int u = __ldg(&inter[idx].user);
    int t = 0;
    neg[idx] = bpr_negative(key, (uint32_t)idx, seen, __ldg(seen_off + u), __ldg(seen_off + u + 1), n_item, &t);
    if (tries) tries[idx] = t;
  }
}

}  // namespace
}  // namespace ure

extern "C" int ure_bpr_negatives(const ure_inter_t* d_inter, int32_t n, int32_t n_item, const int64_t* d_seen_off,
                                 const int32_t* d_seen_items, uint32_t perm_seed, int32_t shard_id, int32_t epoch,
                                 int32_t* d_neg, int32_t* d_tries, void* stream) {
  using namespace ure;
  URE_REQUIRE(n >= 0 && n_item >= 1 && epoch >= 0, URE_EINVAL, "ure_bpr_negatives: n=%d n_item=%d epoch=%d", n,
              n_item, epoch);
  if (n == 0) return 0;
  URE_REQUIRE(d_inter && d_seen_off && d_seen_items && d_neg, URE_EINVAL, "ure_bpr_negatives: null argument");
  const int blocks = (int)((n + 255) / 256 < 4 * num_sms() ? (n + 255) / 256 : 4 * num_sms());
  bpr_negatives_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      d_inter, n, (uint32_t)n_item, d_seen_off, d_seen_items, perm_key(perm_seed, (uint32_t)shard_id, (uint32_t)epoch),
      d_neg, d_tries);
  URE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int ure_mf_train_bpr(const ure_mf_shard_t* d_shards, const ure_bpr_shard_t* d_bpr, int n_shards,
                                const ure_mf_hparams_t* h_hp, int epochs, int64_t step_begin, int64_t step_end,
                                int warps_group0, void* d_workspace, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_shards && d_bpr && h_hp && d_workspace, URE_EINVAL, "ure_mf_train_bpr: null argument");
  URE_REQUIRE(n_shards >= 1 && n_shards <= URE_MAX_SHARDS, URE_EINVAL,
              "ure_mf_train_bpr: n_shards=%d outside [1,%d]", n_shards, URE_MAX_SHARDS);
  URE_REQUIRE(h_hp->batch > 0 && h_hp->lr_step > 0 && epochs > 0, URE_EINVAL,
              "ure_mf_train_bpr: batch/lr_step/epochs must be positive");
  URE_REQUIRE(h_hp->mode == URE_MF_DENSE, URE_EUNSUPPORTED,
              "ure_mf_train_bpr: mode=%d; BPR trains with the DENSE schedule only", h_hp->mode);
  URE_REQUIRE(warps_group0 >= 1 && warps_group0 <= kThreads / 32, URE_EINVAL,
              "ure_mf_train_bpr: warps_group0=%d outside [1,%d]", warps_group0, kThreads / 32);
  return dense<kBpr>(d_shards, n_shards, *h_hp, epochs, step_begin, step_end, warps_group0, d_workspace, d_bpr,
                     stream, "ure_mf_train_bpr");
}
