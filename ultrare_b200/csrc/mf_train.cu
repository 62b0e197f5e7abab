// Fused Matrix-Factorization training (ure_mf_train): the DENSE schedule of mf_dense.cuh with the reference's
// squared-error objective, and the dispatch to the LAZY / OWNER / RUNS schedules.
#include "mf_dense.cuh"

namespace ure {
int g_force_warps_g0 = -1;
}  // namespace ure

extern "C" int64_t ure_mf_train_workspace_bytes(void) {
  const int64_t a = (int64_t)sizeof(ure::Workspace), b = ure::mf_owner_workspace_bytes();
  return a > b ? a : b;
}

extern "C" int ure_mf_train(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* h_hp,
                            int epochs, int64_t step_begin, int64_t step_end, int warps_group0,
                            void* d_workspace, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_shards && h_hp && d_workspace, URE_EINVAL, "ure_mf_train: null argument");
  URE_REQUIRE(n_shards >= 1 && n_shards <= URE_MAX_SHARDS, URE_EINVAL,
              "ure_mf_train: n_shards=%d outside [1,%d]", n_shards, URE_MAX_SHARDS);
  URE_REQUIRE(h_hp->batch > 0 && h_hp->lr_step > 0 && epochs > 0, URE_EINVAL,
              "ure_mf_train: batch/lr_step/epochs must be positive");
  URE_REQUIRE(h_hp->mode >= URE_MF_DENSE && h_hp->mode <= URE_MF_RUNS, URE_EINVAL, "ure_mf_train: mode=%d unknown",
              h_hp->mode);
  if (h_hp->mode == URE_MF_RUNS)
    return mf_train_runs(d_shards, n_shards, h_hp, epochs, step_begin, step_end, d_workspace,
                         static_cast<cudaStream_t>(stream));
  if (h_hp->mode == URE_MF_OWNER)
    return mf_train_owner(d_shards, n_shards, h_hp, epochs, step_begin, step_end, d_workspace,
                          static_cast<cudaStream_t>(stream));
  if (h_hp->mode == URE_MF_LAZY)
    return mf_train_lazy(d_shards, n_shards, h_hp, epochs, step_begin, step_end, d_workspace,
                         static_cast<cudaStream_t>(stream));
  URE_REQUIRE(warps_group0 >= 1 && warps_group0 <= kThreads / 32, URE_EINVAL,
              "ure_mf_train: warps_group0=%d outside [1,%d]", warps_group0, kThreads / 32);
  return dense<kMse>(d_shards, n_shards, *h_hp, epochs, step_begin, step_end, warps_group0, d_workspace, nullptr,
                     stream, "ure_mf_train");
}

// Diagnostics: the next ure_mf_train calls on this workspace record, for their first `steps` steps, six
// SM-clock stamps per CTA (step start, gradients issued, arrive-1 overlap done, barrier 1 passed, sweep
// issued, barrier 2 passed) into d_trace [steps][grid][6] int64.  d_trace = NULL switches tracing off.
extern "C" int ure_mf_train_trace(void* d_workspace, int64_t* d_trace, int steps, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_workspace, URE_EINVAL, "ure_mf_train_trace: null workspace");
  auto* ws = static_cast<Workspace*>(d_workspace);
  long long* p = reinterpret_cast<long long*>(d_trace);
  URE_CUDA(cudaMemcpyAsync(&ws->trace, &p, sizeof(p), cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream)));
  URE_CUDA(cudaMemcpyAsync(&ws->trace_steps, &steps, sizeof(int), cudaMemcpyHostToDevice,
                           static_cast<cudaStream_t>(stream)));
  // the owner schedule keeps its own (disjoint) trace fields in the same workspace
  return mf_owner_trace(d_workspace, p, steps, static_cast<cudaStream_t>(stream));
}

extern "C" int ure_mf_debug_flags(void* d_workspace, unsigned flags, void* stream) {
  using namespace ure;
  URE_REQUIRE(d_workspace, URE_EINVAL, "ure_mf_debug_flags: null workspace");
  auto* ws = static_cast<Workspace*>(d_workspace);
  g_force_warps_g0 = (int)((flags >> 8) & 63u) ? (int)((flags >> 8) & 63u) : -1;
  URE_CUDA(cudaMemcpyAsync(&ws->debug_flags, &flags, sizeof(flags), cudaMemcpyHostToDevice,
                           static_cast<cudaStream_t>(stream)));
  URE_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  return 0;
}

extern "C" int ure_mf_grid_size(void) { return ure::num_sms(); }

extern "C" int ure_mf_flush(const ure_mf_shard_t* h_shards, int n_shards, const ure_mf_hparams_t* h_hp, int epochs,
                            int64_t step_now, void* stream) {
  using namespace ure;
  URE_REQUIRE(h_hp, URE_EINVAL, "ure_mf_flush: null hparams");
  if (h_hp->mode != URE_MF_LAZY) return 0;   // dense / owner schedules: every row is always current
  return mf_flush_lazy(h_shards, n_shards, h_hp, epochs, step_now, static_cast<cudaStream_t>(stream));
}
