// Shared device/host helpers for the ultrare_b200 kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/ultrare_b200.h"

namespace ure {

// ---------------------------------------------------------------- error plumbing
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
int num_sms();

// lazy variant of the MF training step (mf_train_lazy.cu)
int mf_train_lazy(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* hp, int epochs,
                  long long step_begin, long long step_end, void* d_workspace, cudaStream_t st);
int mf_flush_lazy(const ure_mf_shard_t* h_shards, int n_shards, const ure_mf_hparams_t* hp, int epochs,
                  long long step_now, cudaStream_t st);

// owner-computes for tables in HBM (mf_train_runs.cu)
int mf_train_runs(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* hp, int epochs,
                  long long step_begin, long long step_end, void* d_workspace, cudaStream_t st);

// owner-computes variant (mf_train_owner.cu)
int mf_train_owner(const ure_mf_shard_t* d_shards, int n_shards, const ure_mf_hparams_t* hp, int epochs,
                   long long step_begin, long long step_end, void* d_workspace, cudaStream_t st);
int64_t mf_owner_workspace_bytes();
int mf_owner_trace(void* d_workspace, long long* d_trace, int steps, cudaStream_t st);

#define URE_CUDA(call)                                      \
  do {                                                      \
    cudaError_t e__ = (call);                               \
    if (e__ != cudaSuccess) return ::ure::cuda_fail(e__, #call); \
  } while (0)

#define URE_REQUIRE(cond, code, ...)  \
  do {                                \
    if (!(cond)) {                    \
      ::ure::set_error(__VA_ARGS__);  \
      return (code);                  \
    }                                 \
  } while (0)

// ---------------------------------------------------------------- memory ops
// L2-only loads: tables are rewritten by other SMs between grid barriers, L1 is not coherent.
__device__ __forceinline__ float4 ld_cg_f4(const float* p) {
  return __ldcg(reinterpret_cast<const float4*>(p));
}
__device__ __forceinline__ void st_cg_f4(float* p, float4 v) {
  __stcg(reinterpret_cast<float4*>(p), v);
}
// streaming (read-once) 16-byte load that does not pollute L1
__device__ __forceinline__ int4 ld_stream_i4(const void* p) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
// fire-and-forget 16-byte vector reduction into L2 (sm_90+): one LTS atomic per 4 floats
__device__ __forceinline__ void red_add_f4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d)
               : "memory");
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------- grid barrier
// Monotonic-counter barrier for cooperative (co-resident) launches.  `target` is a
// per-thread running value; the counter only grows, so no reset race exists.
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned& target) {
  __syncthreads();
  target += gridDim.x;
  if (threadIdx.x == 0) {
    __threadfence();
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
    while (ld_acquire_u32(counter) < target) {
    }
    __threadfence();
  }
  __syncthreads();
}

}  // namespace ure
