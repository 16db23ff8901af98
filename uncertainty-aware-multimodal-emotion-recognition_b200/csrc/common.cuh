// Shared helpers for libdeer_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>

#include "../../include/deer_b200.h"

namespace deer {

extern std::atomic<long long> g_launches;
extern std::atomic<long long> g_engine_calls[8];
void set_error(const char* fmt, ...);

inline int cuda_status(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return DEER_OK;
  set_error("%s: %s", what, cudaGetErrorString(e));
  return -(1000 + (int)e);
}

#define DEER_CHECK_ARG(cond, msg)                   \
  do {                                              \
    if (!(cond)) {                                  \
      deer::set_error("invalid argument: %s", msg); \
      return DEER_ERR_INVALID;                      \
    }                                               \
  } while (0)

// Programmatic dependent launch: every kernel of the library starts with DEER_PDL_ENTRY() -- it lets the NEXT kernel in
// the stream be scheduled as soon as all CTAs of this one are resident (launch latency, block scheduling, barrier /
// TMEM / tensormap prologues overlap this kernel's tail) and then waits until every kernel it depends on has completed
// and flushed its memory.  Nothing may touch global memory before the wait.  A step is ~300 dependent launches, most
// of them a few microseconds long, so the kernel-to-kernel gap is a first-order cost (DESIGN.md section 7).
#define DEER_PDL_ENTRY()                                         \
  do {                                                           \
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); \
    asm volatile("griddepcontrol.wait;" ::: "memory");           \
  } while (0)

extern int g_pdl;  // deer_set_option(DEER_OPT_PDL): 1 = launch with programmatic stream serialization (default 0)

template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                 Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = g_pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Count + launch + report (no synchronisation: errors here are launch-configuration errors).
#define DEER_LAUNCH(kernel, grid, block, smem, stream, ...)                                              \
  do {                                                                                                   \
    cudaError_t _e = deer::launch_kernel(kernel, dim3(grid), dim3(block), (size_t)(smem),                \
                                         (cudaStream_t)(stream), __VA_ARGS__);                           \
    deer::g_launches.fetch_add(1, std::memory_order_relaxed);                                            \
    if (_e == cudaSuccess) _e = cudaGetLastError();                                                      \
    if (_e != cudaSuccess) return deer::cuda_status(_e, #kernel);                                        \
  } while (0)

constexpr int kNumSMs = 148;  // B200

__host__ __device__ inline long long cdiv(long long a, long long b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------- device math
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// block-wide sum; `red` is >= 32 floats of shared memory; result valid in all threads
__device__ __forceinline__ float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float r = (lane < nw) ? red[lane] : 0.f;
  r = warp_sum(r);
  return r;
}

// per-utterance lengths (packed-sequence semantics): sample b's valid frames are t < clamp(lengths[b], 1, T), lengths
// [B] int32 or int64 (i64 != 0) in device memory, never checked on the host
__device__ __forceinline__ int seq_length(const void* lengths, int i64, int b, int T) {
  const long long L = i64 ? static_cast<const long long*>(lengths)[b] : static_cast<const int*>(lengths)[b];
  return (int)(L < 1 ? 1 : (L > T ? T : L));
}
// row m of a batch-major [B*T, .] layout is (b = m / T, t = m % T): a frame of its utterance (t < L_b), not padding
__device__ __forceinline__ bool seq_row_valid(long long m, const void* lengths, int i64, int T) {
  const int b = (int)(m / T);
  return (int)(m - (long long)b * T) < seq_length(lengths, i64, b, T);
}

// accurate fp32 sigmoid / tanh on the MUFU pipe (ex2 + rcp): |rel err| ~ 2 ulp
__device__ __forceinline__ float sigmoid_f(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float tanh_f(float x) {
  // 1 - 2/(1+e^{2x}); saturates cleanly for |x| large
  const float e = __expf(2.f * x);
  return 1.f - __fdividef(2.f, 1.f + e);
}
// torch F.softplus(beta=1, threshold=20)
__device__ __forceinline__ float softplus_f(float x) { return x > 20.f ? x : log1pf(expf(x)); }
__device__ __forceinline__ float softplus_grad_f(float x) { return x > 20.f ? 1.f : 1.f / (1.f + expf(-x)); }

// digamma for x >= ~0.5 (alpha >= 1 on this path): recurrence to x>=6 then asymptotic series
__device__ __forceinline__ float digamma_f(float x) {
  float r = 0.f;
  while (x < 6.f) {
    r -= 1.f / x;
    x += 1.f;
  }
  const float ix = 1.f / x, ix2 = ix * ix;
  // ln x - 1/2x - 1/12x^2 + 1/120x^4 - 1/252x^6 + 1/240x^8
  const float s = ix2 * (-1.f / 12.f + ix2 * (1.f / 120.f + ix2 * (-1.f / 252.f + ix2 * (1.f / 240.f))));
  return r + logf(x) - 0.5f * ix + s;
}

__device__ __forceinline__ float act_apply(float v, int act) {
  switch (act) {
    case DEER_ACT_RELU: return fmaxf(v, 0.f);
    case DEER_ACT_TANH: return tanhf(v);
    case DEER_ACT_SIGMOID: return 1.f / (1.f + expf(-v));
    default: return v;
  }
}
// out-of-line 4-wide activation for GEMM epilogues: the common case (no activation) never enters it and the libm
// slow paths of tanhf/expf stay out of the unrolled store loops (instruction-cache footprint)
static __device__ __noinline__ float4 act_apply4(float4 v, int act) {
  v.x = act_apply(v.x, act);
  v.y = act_apply(v.y, act);
  v.z = act_apply(v.z, act);
  v.w = act_apply(v.w, act);
  return v;
}
static __device__ __noinline__ float act_apply1(float v, int act) { return act_apply(v, act); }
// derivative expressed through the activation OUTPUT y
__device__ __forceinline__ float act_grad_from_out(float y, int act) {
  switch (act) {
    case DEER_ACT_RELU: return y > 0.f ? 1.f : 0.f;
    case DEER_ACT_TANH: return 1.f - y * y;
    case DEER_ACT_SIGMOID: return y * (1.f - y);
    default: return 1.f;
  }
}

// ------------------------------------------------------------------ Philox-4x32-10
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}

}  // namespace deer
