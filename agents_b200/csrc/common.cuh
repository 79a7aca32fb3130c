// Shared device/host helpers for libb200rl (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/b200rl.h"

namespace b200rl {

// ---- error plumbing ---------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define B200RL_CHECK_ARG(cond, ...)          \
  do {                                       \
    if (!(cond)) {                           \
      ::b200rl::set_error(__VA_ARGS__);      \
      return B200RL_ERR_INVALID;             \
    }                                        \
  } while (0)

#define B200RL_CHECK_LAUNCH(name)                                                   \
  do {                                                                              \
    cudaError_t e__ = cudaGetLastError();                                           \
    if (e__ != cudaSuccess) {                                                       \
      ::b200rl::set_error("%s: CUDA launch failed: %s", name, cudaGetErrorString(e__)); \
      return B200RL_ERR_CUDA;                                                       \
    }                                                                               \
    ::b200rl::count_launch();                                                       \
  } while (0)

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

// ---- programmatic dependent launch (PDL) ---------------------------------------------------
// Every kernel of the library starts with pdl_prologue(): `griddepcontrol.wait` blocks until the
// grids this launch depends on have completed and flushed their memory (a no-op for launches
// without the attribute), then `griddepcontrol.launch_dependents` lets the NEXT kernel of the
// stream be scheduled while this one runs.  With the wait first, ordering is exactly stream
// order; what is gained is that the next grid's launch latency and block scheduling overlap this
// grid's execution instead of following it (2-3 us per node in a captured step).
// Kernels with a global-memory-free prologue (tc2_gemm: barrier init, TMEM allocation) call
// pdl_launch_dependents() first and pdl_wait() after the prologue instead.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ void pdl_prologue() {
  pdl_wait();
  pdl_launch_dependents();
}

// 1 when launches carry cudaLaunchAttributeProgrammaticStreamSerialization (B200RL_PDL, b200rl_set_pdl)
int pdl_enabled();

template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                            cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  if (pdl_enabled()) {
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  }
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<Args&&>(args)...);
}
// Launch errors are picked up by the B200RL_CHECK_LAUNCH that follows every launch.
#define B200RL_LAUNCH(kernel, grid, block, smem, st, ...) \
  (void)::b200rl::launch_k(kernel, dim3(grid), dim3(block), (size_t)(smem), st, __VA_ARGS__)

// ---- Philox4x32-10 (Salmon et al. 2011), the counter-based generator of this library -----
// counter = (elem_lo, elem_hi, call_lo, call_hi), key = (seed_lo, seed_hi).
// oracle/philox.py restates exactly this; tests/test_philox.py pins both against the
// Random123 known-answer vectors.
struct Philox4 {
  uint32_t x, y, z, w;
};

__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint64_t elem, uint64_t call,
                                                           uint64_t seed) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
  uint32_t c0 = (uint32_t)elem, c1 = (uint32_t)(elem >> 32);
  uint32_t c2 = (uint32_t)call, c3 = (uint32_t)(call >> 32);
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = mulhi32(M0, c0), lo0 = M0 * c0;
    uint32_t hi1 = mulhi32(M1, c2), lo1 = M1 * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0;
    uint32_t n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += W0; k1 += W1;
  }
  return Philox4{c0, c1, c2, c3};
}

// uniform int64 in [lo, hi): lo + u64 % (hi-lo)  (TF's int64 uniform also reduces by modulo).
__host__ __device__ __forceinline__ int64_t uniform_i64(uint32_t a, uint32_t b, int64_t lo,
                                                         int64_t hi) {
  uint64_t u = ((uint64_t)b << 32) | (uint64_t)a;
  uint64_t range = (uint64_t)(hi - lo);
  return lo + (int64_t)(u % range);
}
// uniform f32 in [0,1) with 24 random bits.
__host__ __device__ __forceinline__ float uniform_f32(uint32_t a) {
  return (float)(a >> 8) * (1.0f / 16777216.0f);
}

// ---- 16-byte streaming copies -------------------------------------------------------------
__device__ __forceinline__ int4 ld_stream16(const void* p) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream16(void* p, const int4& v) {
  asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x),
               "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum (blockDim.x multiple of 32, <= 1024). Deterministic order.
__device__ __forceinline__ float block_sum(float v, float* smem32) {
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) smem32[wid] = v;
  __syncthreads();
  int nw = (blockDim.x + 31) >> 5;
  float r = (threadIdx.x < nw) ? smem32[threadIdx.x] : 0.f;
  if (wid == 0) r = warp_sum(r);
  if (threadIdx.x == 0) smem32[0] = r;
  __syncthreads();
  r = smem32[0];
  return r;
}

}  // namespace b200rl
