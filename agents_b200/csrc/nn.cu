// Dense / Conv2D forward + backward in true fp32 (kernel family iii, network part).
//
// The reference runs these through Keras -> TensorFlow CPU kernels (Eigen fp32):
//   networks/encoding_network.py:224-312 (conv + dense stack), q_network.py:126-135 (Q head),
//   examples/dqn/mnih15/dqn_train_eval_atari.py:104-110 (the Atari net incl. cast+/255).
// North-star parity is 1e-5 relative on the loss, which BF16/TF32 MMA cannot hold over a
// 3136-wide reduction (SURVEY.md §7 "hard parts"), so this file is a register-tiled fp32 FFMA
// GEMM with pluggable operand views:
//   ARow  A(m,k)=X[m*ld+k]              dense forward, dX = dZ @ W^T
//   ACol  A(m,k)=X[k*ld+m]              dW = X^T @ dZ
//   AConv A(m,k)=im2col(X)(m,k)         implicit-GEMM conv forward (u8 or f32 input, fused
//                                       cast * scale of the reference's preprocessing layer)
//   AConvT A(m,k)=im2col(X)(k,m)        conv filter gradient
//   BRow  B(k,n)=W[k*ld+n]   BCol  B(k,n)=W[n*ld+k]
// Small output grids (fc layers, filter gradients) use deterministic split-K: partial tiles
// go to the caller's workspace and a second kernel reduces them in fixed order and applies
// bias + activation, so results are run-to-run bit-stable.
#include <cuda.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <mutex>
#include <tuple>

#include "common.cuh"

namespace b200rl {

struct FastDiv {
  uint32_t d, mul, shr;
  __host__ FastDiv() : d(1), mul(0), shr(0) {}
  __host__ explicit FastDiv(uint32_t div) : d(div) {
    // round-up magic number method, valid for n < 2^31
    if (div == 1) { mul = 0; shr = 0; return; }
    uint32_t l = 0;
    while ((1u << l) < div) ++l;
    uint64_t m = ((1ull << 32) * ((1ull << l) - div)) / div + 1;
    mul = (uint32_t)m;
    shr = l;
  }
  __device__ __forceinline__ uint32_t div(uint32_t n) const {
    if (d == 1) return n;
    uint32_t t = __umulhi(mul, n);
    return (t + ((n - t) >> 1)) >> (shr - 1);
  }
  __device__ __forceinline__ void divmod(uint32_t n, uint32_t& q, uint32_t& r) const {
    q = div(n);
    r = n - q * d;
  }
};

// Operand views.  Every view is separable: element (row, k) lives at row_off(row) + k_off(k),
// where "row" is m for A views and n for B views.  kKContig says which index is contiguous in
// memory.  `at` is the scalar accessor of the fp32 FFMA kernel; `addr` is the raw address the
// tensor-core kernel copies 16-byte chunks from (tc2_gemm.cuh).
struct ARow {
  const float* p;
  int64_t ld;
  static constexpr bool kKContig = true;
  static constexpr bool kTma2D = true;        // plain row-major [rows, K] matrix: TMA tile loads in tc2
  static constexpr bool kLinearK = true;      // k_off(k) == k * k_stride()
  static constexpr bool kExact = false;
  __device__ __forceinline__ float at(int64_t m, int64_t k) const { return p[m * ld + k]; }
  __device__ __forceinline__ int64_t row_off(int64_t m) const { return m * ld; }
  __device__ __forceinline__ int64_t k_off(int64_t k) const { return k; }
  __device__ __forceinline__ int64_t k_stride() const { return 1; }
  __device__ __forceinline__ const void* addr(int64_t off) const { return p + off; }
};
struct ACol {
  const float* p;
  int64_t ld;
  static constexpr bool kKContig = false;
  static constexpr bool kTma2D = false;
  static constexpr bool kLinearK = true;      // k_off(k) == k * k_stride()
  static constexpr bool kExact = false;
  __device__ __forceinline__ float at(int64_t m, int64_t k) const { return p[k * ld + m]; }
  __device__ __forceinline__ int64_t row_off(int64_t m) const { return m; }
  __device__ __forceinline__ int64_t k_off(int64_t k) const { return k * ld; }
  __device__ __forceinline__ int64_t k_stride() const { return ld; }
  __device__ __forceinline__ const void* addr(int64_t off) const { return p + off; }
};
struct BRow {  // B(k, n) = p[k*ld + n]  (n contiguous)
  const float* p;
  int64_t ld;
  static constexpr bool kNContig = true;
  static constexpr bool kKContig = false;
  static constexpr bool kTma2D = false;
  static constexpr bool kLinearK = true;      // k_off(k) == k * k_stride()
  static constexpr bool kExact = false;
  __device__ __forceinline__ float at(int64_t k, int64_t n) const { return p[k * ld + n]; }
  __device__ __forceinline__ int64_t row_off(int64_t n) const { return n; }
  __device__ __forceinline__ int64_t k_off(int64_t k) const { return k * ld; }
  __device__ __forceinline__ int64_t k_stride() const { return ld; }
  __device__ __forceinline__ const void* addr(int64_t off) const { return p + off; }
};
struct BCol {  // B(k, n) = p[n*ld + k]  (k contiguous)
  const float* p;
  int64_t ld;
  static constexpr bool kNContig = false;
  static constexpr bool kKContig = true;
  static constexpr bool kTma2D = true;        // plain row-major [rows, K] matrix: TMA tile loads in tc2
  static constexpr bool kLinearK = true;      // k_off(k) == k * k_stride()
  static constexpr bool kExact = false;
  __device__ __forceinline__ float at(int64_t k, int64_t n) const { return p[n * ld + k]; }
  __device__ __forceinline__ int64_t row_off(int64_t n) const { return n * ld; }
  __device__ __forceinline__ int64_t k_off(int64_t k) const { return k; }
  __device__ __forceinline__ int64_t k_stride() const { return 1; }
  __device__ __forceinline__ const void* addr(int64_t off) const { return p + off; }
};

struct ConvGeom {
  int H, W, C, KH, KW, F, stride, OH, OW;
  FastDiv d_ohow, d_ow, d_kwc;
  int64_t in_row;   // W*C
  int64_t in_img;   // elements between consecutive images
};

template <typename T>
__device__ __forceinline__ float cvt_in(T v, float scale);
template <>
__device__ __forceinline__ float cvt_in<float>(float v, float) { return v; }
template <>
__device__ __forceinline__ float cvt_in<uint8_t>(uint8_t v, float scale) {
  // tf.cast(obs, f32) / 255 is restated as a division to stay bit-identical to the oracle.
  return __fdiv_rn((float)v, scale);
}

// im2col view: pos = (n, oy, ox), patch = (ky, kx, c) with c fastest (Keras HWIO order).
template <typename T>
struct ConvView {
  const T* x;
  ConvGeom g;
  float scale;
  __device__ __forceinline__ int64_t pos_offset(uint32_t pos) const {
    uint32_t n, r, oy, ox;
    g.d_ohow.divmod(pos, n, r);
    g.d_ow.divmod(r, oy, ox);
    return (int64_t)n * g.in_img + (int64_t)(oy * g.stride) * g.in_row +
           (int64_t)(ox * g.stride) * g.C;
  }
  __device__ __forceinline__ int64_t patch_offset(uint32_t kidx) const {
    uint32_t ky, r;
    g.d_kwc.divmod(kidx, ky, r);
    return (int64_t)ky * g.in_row + r;
  }
  __device__ __forceinline__ float load(int64_t off) const { return cvt_in<T>(x[off], scale); }
};
// fp32 im2col views of an fp32 or uint8 input (the latter with the reference's cast / scale).
// `addr` hands the tensor-core kernel fp32 data, so it only compiles for T = float: uint8 inputs
// reach that kernel through the raw views below.
template <typename T>
struct AConv {
  ConvView<T> v;
  static constexpr bool kKContig = true;
  static constexpr bool kTma2D = false;
  static constexpr bool kLinearK = false;
  static constexpr bool kExact = false;
  __device__ __forceinline__ float at(int64_t m, int64_t k) const {
    return v.load(v.pos_offset((uint32_t)m) + v.patch_offset((uint32_t)k));
  }
  __device__ __forceinline__ int64_t row_off(int64_t m) const { return v.pos_offset((uint32_t)m); }
  __device__ __forceinline__ int64_t k_off(int64_t k) const { return v.patch_offset((uint32_t)k); }
  __device__ __forceinline__ const float* addr(int64_t off) const { return v.x + off; }
};
template <typename T>
struct AConvT {
  ConvView<T> v;
  static constexpr bool kKContig = false;
  static constexpr bool kTma2D = false;
  static constexpr bool kLinearK = false;
  static constexpr bool kExact = false;
  __device__ __forceinline__ float at(int64_t m, int64_t k) const {
    return v.load(v.pos_offset((uint32_t)k) + v.patch_offset((uint32_t)m));
  }
  __device__ __forceinline__ int64_t row_off(int64_t m) const { return v.patch_offset((uint32_t)m); }
  __device__ __forceinline__ int64_t k_off(int64_t k) const { return v.pos_offset((uint32_t)k); }
  __device__ __forceinline__ const float* addr(int64_t off) const { return v.x + off; }
};

// Raw uint8 pixel views for the tensor-core kernel: values 0..255 are exact in TF32, the 1/scale of
// the reference's cast+/255 layer is applied to the accumulator in the epilogue instead.  They
// have no `at`, so they cannot be compiled into the FFMA kernel.
struct AConvU8Raw {
  ConvView<uint8_t> v;
  static constexpr bool kKContig = true;
  static constexpr bool kTma2D = false;
  static constexpr bool kLinearK = false;
  static constexpr bool kExact = true;
  __device__ __forceinline__ int64_t row_off(int64_t m) const { return v.pos_offset((uint32_t)m); }
  __device__ __forceinline__ int64_t k_off(int64_t k) const { return v.patch_offset((uint32_t)k); }
  __device__ __forceinline__ const void* addr(int64_t off) const { return v.x + off; }
};
struct AConvTU8Raw {
  ConvView<uint8_t> v;
  static constexpr bool kKContig = false;
  static constexpr bool kTma2D = false;
  static constexpr bool kLinearK = false;
  static constexpr bool kExact = true;
  __device__ __forceinline__ int64_t row_off(int64_t m) const { return v.patch_offset((uint32_t)m); }
  __device__ __forceinline__ int64_t k_off(int64_t k) const { return v.pos_offset((uint32_t)k); }
  __device__ __forceinline__ const void* addr(int64_t off) const { return v.x + off; }
};

__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == B200RL_ACT_RELU) return fmaxf(v, 0.f);
  if (act == B200RL_ACT_TANH) return tanhf(v);
  return v;
}

// Input-gradient mask: when the GEMM input X is the OUTPUT of an activation (the previous layer
// of the stack), dLoss/dX is multiplied by act'(X) on its way out, so the caller receives the
// gradient w.r.t. that layer's pre-activation and the separate act_bwd pass disappears.
struct ActMask {
  const float* y = nullptr;   // X as produced by the previous layer (nullptr: no mask)
  int64_t ld = 0;             // dense: row stride of y; conv: elements between images
  int act = 0;
};
__device__ __forceinline__ float dact(float y, float g, int act) {
  if (act == B200RL_ACT_RELU) return y > 0.f ? g : 0.f;
  if (act == B200RL_ACT_TANH) return g * (1.f - y * y);
  return g;
}

}  // namespace b200rl
#include "tc2_gemm.cuh"
namespace b200rl {

constexpr int BK = 16;

// C[M,N] (+)= act(A @ B + bias)   or   ws[split] = partial(A @ B) when splits > 1.
template <int BM, int BN, int TM, int TN, class AL, class BL>
__global__ void __launch_bounds__(256) sgemm_kernel(const AL a, const BL b, float* __restrict__ C,
                                                    const float* __restrict__ bias, int64_t M,
                                                    int64_t N, int64_t K, int act, int beta,
                                                    int splits, int64_t k_per_split,
                                                    float* __restrict__ ws, const ActMask mask) {
  pdl_prologue();
  static_assert((BM / TM) * (BN / TN) == 256, "thread grid must be 256");
  constexpr int TX = BN / TN;
  constexpr int GM = TM >= 4 ? 4 : TM, GN = TN >= 4 ? 4 : TN;  // contiguous group widths
  constexpr int NGM = TM / GM, NGN = TN / GN;
  constexpr int APT = BM * BK / 256, BPT = BN * BK / 256;  // elements per thread per tile
  __shared__ __align__(16) float As[2][BK][BM + 4];
  __shared__ __align__(16) float Bs[2][BK][BN + 4];

  const int tid = threadIdx.x;
  const int tx = tid % TX, ty = tid / TX;
  const int64_t m0 = (int64_t)blockIdx.y * BM, n0 = (int64_t)blockIdx.x * BN;
  const int split = blockIdx.z;
  const int64_t kb = (int64_t)split * k_per_split;
  const int64_t ke = (kb + k_per_split < K) ? kb + k_per_split : K;

  // tile-load coordinates
  int a_m[APT], a_k[APT], b_n[BPT], b_k[BPT];
#pragma unroll
  for (int i = 0; i < APT; ++i) {
    if (AL::kKContig) { a_k[i] = tid % BK; a_m[i] = tid / BK + i * (256 / BK); }
    else { a_m[i] = tid % BM; a_k[i] = tid / BM + i * (256 / BM); }
  }
#pragma unroll
  for (int i = 0; i < BPT; ++i) {
    if (BL::kNContig) { b_n[i] = tid % BN; b_k[i] = tid / BN + i * (256 / BN); }
    else { b_k[i] = tid % BK; b_n[i] = tid / BK + i * (256 / BK); }
  }

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  float ra[APT], rb[BPT];
  auto load_tile = [&](int64_t k0) {
#pragma unroll
    for (int i = 0; i < APT; ++i) {
      const int64_t m = m0 + a_m[i], k = k0 + a_k[i];
      ra[i] = (m < M && k < ke) ? a.at(m, k) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < BPT; ++i) {
      const int64_t n = n0 + b_n[i], k = k0 + b_k[i];
      rb[i] = (n < N && k < ke) ? b.at(k, n) : 0.f;
    }
  };
  auto store_tile = [&](int buf) {
#pragma unroll
    for (int i = 0; i < APT; ++i) As[buf][a_k[i]][a_m[i]] = ra[i];
#pragma unroll
    for (int i = 0; i < BPT; ++i) Bs[buf][b_k[i]][b_n[i]] = rb[i];
  };

  int buf = 0;
  if (kb < ke) {
    load_tile(kb);
    store_tile(0);
  }
  __syncthreads();
  for (int64_t k0 = kb; k0 < ke; k0 += BK) {
    const bool has_next = k0 + BK < ke;
    if (has_next) load_tile(k0 + BK);
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float fa[TM], fb[TN];
#pragma unroll
      for (int g = 0; g < NGM; ++g)
#pragma unroll
        for (int i = 0; i < GM; ++i) fa[g * GM + i] = As[buf][kk][g * (BM / NGM) + ty * GM + i];
#pragma unroll
      for (int g = 0; g < NGN; ++g)
#pragma unroll
        for (int j = 0; j < GN; ++j) fb[g * GN + j] = Bs[buf][kk][g * (BN / NGN) + tx * GN + j];
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(fa[i], fb[j], acc[i][j]);
    }
    if (has_next) {
      store_tile(buf ^ 1);
      __syncthreads();
      buf ^= 1;
    }
  }

  float* out = (splits > 1) ? ws + (int64_t)split * M * N : C;
#pragma unroll
  for (int gi = 0; gi < NGM; ++gi)
#pragma unroll
    for (int i = 0; i < GM; ++i) {
      const int64_t m = m0 + gi * (BM / NGM) + ty * GM + i;
      if (m >= M) continue;
#pragma unroll
      for (int gj = 0; gj < NGN; ++gj)
#pragma unroll
        for (int j = 0; j < GN; ++j) {
          const int64_t n = n0 + gj * (BN / NGN) + tx * GN + j;
          if (n >= N) continue;
          float v = acc[gi * GM + i][gj * GN + j];
          if (splits == 1) {
            if (bias) v += bias[n];
            v = apply_act(v, act);
            if (mask.y) v = dact(mask.y[m * mask.ld + n], v, mask.act);
            if (beta) v += out[m * N + n];
          }
          out[m * N + n] = v;
        }
    }
}

__global__ void splitk_reduce_kernel(const float* __restrict__ ws, float* __restrict__ C,
                                     const float* __restrict__ bias, int64_t MN, int64_t N,
                                     int splits, int act, int beta, const ActMask mask) {
  pdl_prologue();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= MN) return;
  float v = 0.f;
  for (int s = 0; s < splits; ++s) v += ws[(int64_t)s * MN + i];
  if (bias) v += bias[i % N];
  v = apply_act(v, act);
  if (mask.y) v = dact(mask.y[(i / N) * mask.ld + i % N], v, mask.act);
  if (beta) v += C[i];
  C[i] = v;
}

// dZ = dY * act'(Y); 16-byte accesses when n and the pointers allow (HBM-bound: 12 B / element)
__global__ void act_bwd_kernel(const float* __restrict__ Y, const float* __restrict__ dY,
                               float* __restrict__ dZ, int64_t n, int act, int vec) {
  pdl_prologue();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (vec) {
    const int64_t n4 = n >> 2;
    for (int64_t i = tid; i < n4; i += stride) {
      const float4 y = reinterpret_cast<const float4*>(Y)[i];
      const float4 g = reinterpret_cast<const float4*>(dY)[i];
      reinterpret_cast<float4*>(dZ)[i] = make_float4(dact(y.x, g.x, act), dact(y.y, g.y, act),
                                                     dact(y.z, g.z, act), dact(y.w, g.w, act));
    }
    return;
  }
  for (int64_t i = tid; i < n; i += stride) dZ[i] = dact(Y[i], dY[i], act);
}

// Column sums of dZ[M,N] in two deterministic stages.
constexpr int kColRows = 512;  // rows per partial block
// Block = 32 columns x 8 row-lanes: a warp reads 128 contiguous bytes of one row, the 8 warps
// walk kColRows rows in an interleaved fashion and are combined through shared memory in a
// fixed order (deterministic).
__global__ void __launch_bounds__(256) colsum_partial_kernel(const float* __restrict__ dZ,
                                                             float* __restrict__ part, int64_t M,
                                                             int64_t N) {
  pdl_prologue();
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t n = (int64_t)blockIdx.x * 32 + lane;
  const int64_t mb = (int64_t)blockIdx.y * kColRows;
  const int64_t me = mb + kColRows < M ? mb + kColRows : M;
  float s = 0.f;
  if (n < N) {
#pragma unroll 4
    for (int64_t m = mb + w; m < me; m += 8) s += dZ[m * N + n];
  }
  red[w][lane] = s;
  __syncthreads();
  if (w == 0 && n < N) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][lane];
    part[(int64_t)blockIdx.y * N + n] = t;
  }
}
__global__ void __launch_bounds__(256) colsum_final_kernel(const float* __restrict__ part,
                                                           float* __restrict__ db, int64_t nparts,
                                                           int64_t N, int beta) {
  pdl_prologue();
  // one warp per column: lanes stride over the partials, fixed-order shuffle reduction
  const int lane = threadIdx.x & 31;
  const int64_t n = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (n >= N) return;
  float s = 0.f;
  for (int64_t p = lane; p < nparts; p += 32) s += part[p * N + n];
  s = warp_sum(s);
  if (lane == 0) db[n] = beta ? db[n] + s : s;
}


// ---------------------------------------------------------------------------------------
// Skinny heads: Dense layers with N <= 16 outputs (Q head, value head, action means).
// A tensor-core tile would be >= 87 % padding and the FFMA tiles need a split-K + reduce pair
// for 256 rows; these three kernels are plain bandwidth-bound sweeps with W staged in shared
// memory.  Used when the GEMM mode is not 0 (their weight gradient accumulates with atomics).
// ---------------------------------------------------------------------------------------
constexpr int kSkinnyMaxN = 16;
constexpr int kSkinnySmem = 48 * 1024;

// Y[m, :] = act(X[m, :] @ W + b): one warp per row, lanes stride over k, N shuffle reductions.
template <int NMAX>
__global__ void __launch_bounds__(256) skinny_fwd_kernel(const float* __restrict__ X, int64_t ldx,
                                                         const float* __restrict__ W,
                                                         const float* __restrict__ bias,
                                                         float* __restrict__ Y, int64_t M, int K,
                                                         int N, int act) {
  pdl_prologue();
  extern __shared__ float sw[];                       // [K, N]
  for (int i = threadIdx.x; i < K * N; i += blockDim.x) sw[i] = W[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int64_t m = (int64_t)blockIdx.x * nw + warp; m < M; m += (int64_t)gridDim.x * nw) {
    float acc[NMAX];
#pragma unroll
    for (int n = 0; n < NMAX; ++n) acc[n] = 0.f;
    const float* x = X + m * ldx;
#pragma unroll 4
    for (int k = lane; k < K; k += 32) {
      const float xv = x[k];
      const float* w = sw + k * N;
#pragma unroll
      for (int n = 0; n < NMAX; ++n)
        if (n < N) acc[n] = fmaf(xv, w[n], acc[n]);
    }
#pragma unroll
    for (int n = 0; n < NMAX; ++n)
      if (n < N) acc[n] = warp_sum(acc[n]);
    if (lane == 0) {
#pragma unroll
      for (int n = 0; n < NMAX; ++n)
        if (n < N) Y[m * N + n] = apply_act(acc[n] + (bias ? bias[n] : 0.f), act);
    }
  }
}

// dX[m, k] = sum_n dY[m, n] W[k, n]  (* act'(X[m, k]) of the producing layer): 4 k per thread.
template <int NMAX>
__global__ void __launch_bounds__(256) skinny_dx_kernel(const float* __restrict__ dY,
                                                        const float* __restrict__ W,
                                                        float* __restrict__ dX, int64_t M, int K,
                                                        int N, const ActMask mask) {
  pdl_prologue();
  extern __shared__ float sw[];                       // [K, N]
  for (int i = threadIdx.x; i < K * N; i += blockDim.x) sw[i] = W[i];
  __syncthreads();
  const int kq = (K + 3) >> 2;                        // k quads per row
  const int64_t total = M * kq;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = i / kq;
    const int k0 = (int)(i - m * kq) * 4;
    float dy[NMAX];
#pragma unroll
    for (int n = 0; n < NMAX; ++n) dy[n] = n < N ? dY[m * N + n] : 0.f;
    float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (k0 + q < K) {
        const float* w = sw + (k0 + q) * N;
#pragma unroll
        for (int n = 0; n < NMAX; ++n)
          if (n < N) o[q] = fmaf(dy[n], w[n], o[q]);
        if (mask.y) o[q] = dact(mask.y[m * mask.ld + k0 + q], o[q], mask.act);
      }
    }
    float* dst = dX + m * K + k0;
    if ((K & 3) == 0) *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
    else
      for (int q = 0; q < 4; ++q)
        if (k0 + q < K) dst[q] = o[q];
  }
}

// dW[k, n] += sum_m X[m, k] dY[m, n], db[n] += sum_m dY[m, n] over the CTA's slab of rows; thread
// t owns input features k = t, t + blockDim, ...; the slab's dY rows are staged in shared memory.
template <int NMAX, int KPT>
__global__ void __launch_bounds__(256) skinny_dw_kernel(const float* __restrict__ X, int64_t ldx,
                                                        const float* __restrict__ dY,
                                                        float* __restrict__ dW,
                                                        float* __restrict__ db, int64_t M, int K,
                                                        int N, int64_t rows_per_cta) {
  pdl_prologue();
  constexpr int kChunk = 64;                          // rows of dY staged per step
  __shared__ float sdy[kChunk * NMAX];
  const int64_t mb = (int64_t)blockIdx.x * rows_per_cta;
  const int64_t me = (mb + rows_per_cta < M) ? mb + rows_per_cta : M;
  float acc[KPT][NMAX];
#pragma unroll
  for (int j = 0; j < KPT; ++j)
#pragma unroll
    for (int n = 0; n < NMAX; ++n) acc[j][n] = 0.f;
  float bsum = 0.f;
  // K < blockDim: the threads form G = blockDim / K' row groups (K' = K rounded up to a warp), group
  // g takes rows g, g + G, ... of every staged chunk (run 12: 100 of 256 threads worked on the PPO
  // heads); the groups meet in the atomics below.
  const int kpad = (K + 31) & ~31;
  const int G = (KPT == 1 && kpad < (int)blockDim.x) ? (int)blockDim.x / kpad : 1;
  const int rg = G > 1 ? (int)threadIdx.x / kpad : 0;
  const int kt = G > 1 ? (int)threadIdx.x - rg * kpad : (int)threadIdx.x;
  const bool live = rg < G;
  for (int64_t m0 = mb; m0 < me; m0 += kChunk) {
    const int rows = (int)((me - m0 < kChunk) ? me - m0 : kChunk);
    __syncthreads();
    for (int i = threadIdx.x; i < rows * N; i += blockDim.x) sdy[(i / N) * NMAX + i % N] = dY[m0 * N + i];
    __syncthreads();
    if ((int)threadIdx.x < N)
      for (int r = 0; r < rows; ++r) bsum += sdy[r * NMAX + threadIdx.x];
#pragma unroll
    for (int j = 0; j < KPT; ++j) {
      const int k = kt + j * blockDim.x;
      if (k < K && live) {
        const float* xp = X + m0 * ldx + k;
        int r = rg;
        for (; r + 3 * G < rows; r += 4 * G) {        // 4 independent loads in flight per thread
          float xv[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) xv[u] = xp[(int64_t)(r + u * G) * ldx];
#pragma unroll
          for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int n = 0; n < NMAX; ++n)
              if (n < N) acc[j][n] = fmaf(xv[u], sdy[(r + u * G) * NMAX + n], acc[j][n]);
        }
        for (; r < rows; r += G) {
          const float xv = xp[(int64_t)r * ldx];
#pragma unroll
          for (int n = 0; n < NMAX; ++n)
            if (n < N) acc[j][n] = fmaf(xv, sdy[r * NMAX + n], acc[j][n]);
        }
      }
    }
  }
  if (G > 1) {
    // the row groups add their sums in a fixed order (a single-CTA launch stays bit-reproducible)
    extern __shared__ float skinny_red[];             // [K, N]
    for (int i = threadIdx.x; i < K * N; i += blockDim.x) skinny_red[i] = 0.f;
    for (int g = 0; g < G; ++g) {
      __syncthreads();
      if (live && rg == g && kt < K) {
#pragma unroll
        for (int n = 0; n < NMAX; ++n)
          if (n < N) skinny_red[kt * N + n] += acc[0][n];
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < K * N; i += blockDim.x) atomicAdd(dW + i, skinny_red[i]);
  } else {
#pragma unroll
    for (int j = 0; j < KPT; ++j) {
      const int k = kt + j * blockDim.x;
      if (k < K && live) {
#pragma unroll
        for (int n = 0; n < NMAX; ++n)
          if (n < N) atomicAdd(dW + (int64_t)k * N + n, acc[j][n]);
      }
    }
  }
  if (db != nullptr && (int)threadIdx.x < N) atomicAdd(db + threadIdx.x, bsum);
}

// ---- thin-input layers (K <= 32: observation -> first hidden layer) ----------------------------
// Run 12 (PPO, 524 288 rows): x[M,17] @ W[17,200] fell through to the first-generation tensor-core
// kernel (K % 4 != 0) at ~900 us and its weight gradient to the FFMA GEMM at ~600 us, against an
// HBM floor of 65 us (the [M,200] activation is written / read once).  Both are one outer product
// per row: thread (cq, rg) owns output columns 4cq..4cq+3 for rows rg*8..rg*8+7 of every 32-row
// chunk; the chunk of X sits in shared memory (broadcast reads), W / dW columns in registers or
// shared memory, the wide operand moves as coalesced float4.
constexpr int kThinMaxK = 32, kThinMaxN = 256, kThinRows = 32;

__global__ void __launch_bounds__(256) thin_fwd_kernel(const float* __restrict__ X, int64_t ldx,
                                                       const float* __restrict__ W,
                                                       const float* __restrict__ bias,
                                                       float* __restrict__ Y, int64_t M, int K,
                                                       int N, int act, int64_t chunks) {
  pdl_prologue();
  extern __shared__ float4 thin_smem[];
  const int KP = (K + 3) & ~3, nq = N >> 2;
  float4* sw = thin_smem;                              // [KP][nq] (rows >= K are zero)
  float* sx = reinterpret_cast<float*>(thin_smem + KP * nq);   // [kThinRows][KP]
  for (int i = threadIdx.x; i < KP * nq; i += blockDim.x)
    sw[i] = (i / nq) < K ? reinterpret_cast<const float4*>(W)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
  const int cq = threadIdx.x & 63, rg = threadIdx.x >> 6;
  const bool active = cq < nq;
  float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (bias && active) b4 = reinterpret_cast<const float4*>(bias)[cq];
  for (int64_t chunk = blockIdx.x; chunk < chunks; chunk += gridDim.x) {
    const int64_t m0 = chunk * kThinRows;
    __syncthreads();
    for (int i = threadIdx.x; i < kThinRows * KP; i += blockDim.x) {
      const int r = i / KP, k = i - r * KP;
      sx[i] = (m0 + r < M && k < K) ? X[(m0 + r) * ldx + k] : 0.f;
    }
    __syncthreads();
    if (!active) continue;
    float4 acc[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) acc[r] = b4;
    for (int k = 0; k < KP; k += 4) {
      const float4 w0 = sw[(k + 0) * nq + cq], w1 = sw[(k + 1) * nq + cq];
      const float4 w2 = sw[(k + 2) * nq + cq], w3 = sw[(k + 3) * nq + cq];
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const float4 x = *reinterpret_cast<const float4*>(sx + (rg * 8 + r) * KP + k);
        acc[r].x = fmaf(x.x, w0.x, acc[r].x); acc[r].y = fmaf(x.x, w0.y, acc[r].y);
        acc[r].z = fmaf(x.x, w0.z, acc[r].z); acc[r].w = fmaf(x.x, w0.w, acc[r].w);
        acc[r].x = fmaf(x.y, w1.x, acc[r].x); acc[r].y = fmaf(x.y, w1.y, acc[r].y);
        acc[r].z = fmaf(x.y, w1.z, acc[r].z); acc[r].w = fmaf(x.y, w1.w, acc[r].w);
        acc[r].x = fmaf(x.z, w2.x, acc[r].x); acc[r].y = fmaf(x.z, w2.y, acc[r].y);
        acc[r].z = fmaf(x.z, w2.z, acc[r].z); acc[r].w = fmaf(x.z, w2.w, acc[r].w);
        acc[r].x = fmaf(x.w, w3.x, acc[r].x); acc[r].y = fmaf(x.w, w3.y, acc[r].y);
        acc[r].z = fmaf(x.w, w3.z, acc[r].z); acc[r].w = fmaf(x.w, w3.w, acc[r].w);
      }
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int64_t m = m0 + rg * 8 + r;
      if (m < M) {
        float4 v = acc[r];
        v.x = apply_act(v.x, act); v.y = apply_act(v.y, act);
        v.z = apply_act(v.z, act); v.w = apply_act(v.w, act);
        reinterpret_cast<float4*>(Y + m * N)[cq] = v;
      }
    }
  }
}

// dW[K,N] += X^T dZ, db[N] += column sums of dZ over the CTA's row range.
template <int KMAX>
__global__ void __launch_bounds__(256, KMAX <= 20 ? 2 : 1) thin_dw_kernel(const float* __restrict__ X, int64_t ldx,
                                                      const float* __restrict__ dZ,
                                                      float* __restrict__ dW,
                                                      float* __restrict__ db, int64_t M, int K,
                                                      int N, int64_t rows_per_cta) {
  pdl_prologue();
  extern __shared__ float4 thin_smem[];
  const int nq = N >> 2;
  float* sx = reinterpret_cast<float*>(thin_smem);     // [kThinRows][KMAX]
  float* sred = sx + kThinRows * KMAX;                 // [(K + 1)][N] cross-row-group sums
  for (int i = threadIdx.x; i < (K + 1) * N; i += blockDim.x) sred[i] = 0.f;
  const int cq = threadIdx.x & 63, rg = threadIdx.x >> 6;
  const bool active = cq < nq;
  float4 acc[KMAX], bsum = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int k = 0; k < KMAX; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  const int64_t mb = (int64_t)blockIdx.x * rows_per_cta;
  const int64_t me = (mb + rows_per_cta < M) ? mb + rows_per_cta : M;
  for (int64_t m0 = mb; m0 < me; m0 += kThinRows) {
    __syncthreads();
    for (int i = threadIdx.x; i < kThinRows * KMAX; i += blockDim.x) {
      const int r = i / KMAX, k = i - r * KMAX;
      sx[i] = (m0 + r < me && k < K) ? X[(m0 + r) * ldx + k] : 0.f;
    }
    __syncthreads();
    if (!active) continue;
#pragma unroll 1
    for (int h = 0; h < 8; h += 4) {                   // two halves of 4 rows: 128 registers, 2 CTAs / SM
    float4 dz[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int64_t m = m0 + rg * 8 + h + r;
      dz[r] = m < me ? reinterpret_cast<const float4*>(dZ + m * N)[cq] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      bsum.x += dz[r].x; bsum.y += dz[r].y; bsum.z += dz[r].z; bsum.w += dz[r].w;
      const float* xr = sx + (rg * 8 + h + r) * KMAX;
#pragma unroll
      for (int k = 0; k < KMAX; k += 4) {
        const float4 x = *reinterpret_cast<const float4*>(xr + k);
        acc[k + 0].x = fmaf(x.x, dz[r].x, acc[k + 0].x); acc[k + 0].y = fmaf(x.x, dz[r].y, acc[k + 0].y);
        acc[k + 0].z = fmaf(x.x, dz[r].z, acc[k + 0].z); acc[k + 0].w = fmaf(x.x, dz[r].w, acc[k + 0].w);
        acc[k + 1].x = fmaf(x.y, dz[r].x, acc[k + 1].x); acc[k + 1].y = fmaf(x.y, dz[r].y, acc[k + 1].y);
        acc[k + 1].z = fmaf(x.y, dz[r].z, acc[k + 1].z); acc[k + 1].w = fmaf(x.y, dz[r].w, acc[k + 1].w);
        acc[k + 2].x = fmaf(x.z, dz[r].x, acc[k + 2].x); acc[k + 2].y = fmaf(x.z, dz[r].y, acc[k + 2].y);
        acc[k + 2].z = fmaf(x.z, dz[r].z, acc[k + 2].z); acc[k + 2].w = fmaf(x.z, dz[r].w, acc[k + 2].w);
        acc[k + 3].x = fmaf(x.w, dz[r].x, acc[k + 3].x); acc[k + 3].y = fmaf(x.w, dz[r].y, acc[k + 3].y);
        acc[k + 3].z = fmaf(x.w, dz[r].z, acc[k + 3].z); acc[k + 3].w = fmaf(x.w, dz[r].w, acc[k + 3].w);
      }
    }
    }
  }
  // the four row groups add their partial sums in a fixed order (a single-CTA launch, i.e. a small
  // batch, is bit-reproducible; larger ones meet in the global atomics below)
  for (int g = 0; g < 4; ++g) {
    __syncthreads();
    if (active && rg == g) {
#pragma unroll
      for (int k = 0; k < KMAX; ++k) {
        if (k < K) {
          float4* d = reinterpret_cast<float4*>(sred + k * N) + cq;
          float4 v = *d;
          v.x += acc[k].x; v.y += acc[k].y; v.z += acc[k].z; v.w += acc[k].w;
          *d = v;
        }
      }
      float4* d = reinterpret_cast<float4*>(sred + K * N) + cq;
      float4 v = *d;
      v.x += bsum.x; v.y += bsum.y; v.z += bsum.z; v.w += bsum.w;
      *d = v;
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < K * N; i += blockDim.x) atomicAdd(dW + i, sred[i]);
  if (db != nullptr)
    for (int i = threadIdx.x; i < N; i += blockDim.x) atomicAdd(db + i, sred[K * N + i]);
}

static int thin_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200RL_THIN");
    v = e ? atoi(e) : 1;
  }
  return v;
}

static int skinny_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200RL_SKINNY");
    v = e ? atoi(e) : 1;
  }
  return v;
}

// col2im in gather form (deterministic): dX[n,y,x,c] = sum over kernel taps hitting (y,x).
__global__ void col2im_kernel(const float* __restrict__ dcol, float* __restrict__ dX, ConvGeom g,
                              int64_t total, int Kc, const ActMask mask) {
  pdl_prologue();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % g.C);
  int64_t r = i / g.C;
  const int x = (int)(r % g.W);
  r /= g.W;
  const int y = (int)(r % g.H);
  const int64_t n = r / g.H;
  float s = 0.f;
  for (int ky = y % g.stride; ky < g.KH && ky <= y; ky += g.stride) {
    const int oy = (y - ky) / g.stride;
    if (oy >= g.OH) continue;
    for (int kx = x % g.stride; kx < g.KW && kx <= x; kx += g.stride) {
      const int ox = (x - kx) / g.stride;
      if (ox >= g.OW) continue;
      const int64_t pos = (n * g.OH + oy) * g.OW + ox;
      s += dcol[pos * Kc + (ky * g.KW + kx) * g.C + c];
    }
  }
  if (mask.y) s = dact(mask.y[n * mask.ld + ((int64_t)y * g.W + x) * g.C + c], s, mask.act);
  dX[i] = s;
}

// ---------------------------------------------------------------------------------------
// host-side dispatch
// ---------------------------------------------------------------------------------------
struct GemmArgs {
  float* C;
  const float* bias;
  int64_t M, N, K;
  int act, beta;
  void* ws;
  int64_t ws_bytes;
  cudaStream_t st;
  float out_scale = 1.f;  // tensor-core path only: multiplies the accumulator (raw-u8 operands)
  ActMask mask{};         // input-gradient GEMMs: multiply the result by act'(mask.y)
};

template <int BM, int BN, int TM, int TN, class AL, class BL>
static int launch_gemm_cfg(const AL& a, const BL& b, const GemmArgs& g) {
  const int64_t tm = (g.M + BM - 1) / BM, tn = (g.N + BN - 1) / BN;
  const int64_t tiles = tm * tn;
  int splits = 1;
  const int64_t target = 2 * kNumSMs;
  if (tiles < target && g.K >= 8 * BK && g.ws != nullptr) {
    int64_t want = (target + tiles - 1) / tiles;
    int64_t max_by_k = g.K / (4 * BK);
    int64_t max_by_ws = g.ws_bytes / (int64_t)(g.M * g.N * sizeof(float));
    int64_t s = want;
    if (s > max_by_k) s = max_by_k;
    if (s > max_by_ws) s = max_by_ws;
    if (s > 65535) s = 65535;
    if (s >= 2) splits = (int)s;
  }
  int64_t kps = (g.K + splits - 1) / splits;
  kps = (kps + BK - 1) / BK * BK;
  splits = (int)((g.K + kps - 1) / kps);
  if (splits < 1) splits = 1;
  B200RL_CHECK_ARG(tm <= 65535, "gemm: M too large for grid.y (%lld tiles)", (long long)tm);
  dim3 grid((unsigned)tn, (unsigned)tm, (unsigned)splits);
  B200RL_LAUNCH((sgemm_kernel<BM, BN, TM, TN, AL, BL>), grid, 256, 0, g.st, a, b, g.C, g.bias, g.M, g.N, g.K, g.act, g.beta, splits, kps, (float*)g.ws, g.mask);
  B200RL_CHECK_LAUNCH("sgemm");
  if (splits > 1) {
    const int64_t MN = g.M * g.N;
    B200RL_LAUNCH(splitk_reduce_kernel, (unsigned)((MN + 255) / 256), 256, 0, g.st, (const float*)g.ws, g.C, g.bias, MN, g.N, splits, g.act, g.beta, g.mask);
    B200RL_CHECK_LAUNCH("splitk_reduce");
  }
  return B200RL_OK;
}

// 0 = fp32 FFMA (sgemm_kernel), 1 = tcgen05 3xTF32, 2 = tcgen05 single-pass TF32 (not 1e-5 safe)
// B200RL_FUSE_BIAS_GRAD=0 keeps the separate column-sum kernels (A/B switch for profiles/)
static int fuse_bias_grad() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200RL_FUSE_BIAS_GRAD");
    v = e ? atoi(e) : 1;
  }
  return v;
}
static int g_gemm_mode = -1;
static int gemm_mode() {
  if (g_gemm_mode < 0) {
    const char* e = getenv("B200RL_GEMM_MODE");
    g_gemm_mode = e ? atoi(e) : 1;
  }
  return g_gemm_mode;
}

// ---- tensor-core (tc2) kernel: eligibility and launch ------------------------------------------
// B200RL_TC2_FLAGS: A/B switches of tc2_gemm.cuh (as b200rl_set_tc2_flags), read at the first launch.
static void tc2_env_flags() {
  static bool done = false;
  if (done) return;
  done = true;
  const char* f = getenv("B200RL_TC2_FLAGS");
  if (f) {
    const int flags = atoi(f);
    cudaMemcpyToSymbol(tc2::g_tc2_flags, &flags, sizeof(flags));
  }
}
// Work distribution of the persistent GEMM: 0 = static striding (a few per cent faster when the
// kernel has the GPU to itself), 1 = dynamic (global counter): CTAs whose SM is busy with a
// collective or a kernel of another stream take fewer tiles instead of delaying the launch.  The
// data-parallel Learner switches it on (run 17, 2 GPUs: 0.93 -> 0.946 weak-scaling efficiency
// together with NCCL_MAX_CTAS=8).
static int g_tile_sched = -1;
static bool tile_scheduler_dynamic() {
  if (g_tile_sched < 0) {
    const char* e = getenv("B200RL_TILE_SCHED");
    g_tile_sched = e ? (atoi(e) != 0) : 0;
  }
  return g_tile_sched != 0;
}
// tc2 only takes operands whose every 16-byte chunk is contiguous and aligned in global memory.
// There is no overload for the fp32-cast uint8 conv views: they never take the tensor route.
static bool al16(const void* p) { return ((uintptr_t)p & 15) == 0; }
static bool tc2_ok(const ARow& v, int64_t rows, int64_t K) { return (v.ld & 3) == 0 && al16(v.p) && (K & 3) == 0; }
static bool tc2_ok(const BCol& v, int64_t rows, int64_t K) { return (v.ld & 3) == 0 && al16(v.p) && (K & 3) == 0; }
static bool tc2_ok(const ACol& v, int64_t rows, int64_t K) { return (v.ld & 3) == 0 && al16(v.p) && (rows & 3) == 0; }
static bool tc2_ok(const BRow& v, int64_t rows, int64_t K) { return (v.ld & 3) == 0 && al16(v.p) && (rows & 3) == 0; }
static bool conv_f32_ok(const ConvView<float>& v) {
  return (v.g.C & 3) == 0 && (v.g.in_img & 3) == 0 && al16(v.x);
}
static bool tc2_ok(const AConv<float>& v, int64_t rows, int64_t K) { return conv_f32_ok(v.v); }
static bool tc2_ok(const AConvT<float>& v, int64_t rows, int64_t K) { return conv_f32_ok(v.v); }
static bool conv_u8_ok(const ConvView<uint8_t>& v) {
  const int64_t kwc = (int64_t)v.g.KW * v.g.C;
  return (kwc & 15) == 0 && (((int64_t)v.g.stride * v.g.C) & 15) == 0 && (v.g.in_row & 15) == 0 &&
         (v.g.in_img & 15) == 0 && al16(v.x);
}
static bool tc2_ok(const AConvU8Raw& v, int64_t rows, int64_t K) { return conv_u8_ok(v.v) && (K & 15) == 0; }
static bool tc2_ok(const AConvTU8Raw& v, int64_t rows, int64_t K) { return conv_u8_ok(v.v) && (rows & 15) == 0; }


// ---- TMA tensor maps for plain 2-D operands (tc2) ---------------------------------------------
// cuTensorMapEncodeTiled is fetched through the runtime (no link against libcuda); maps are cached
// by (base, rows, K, ld, box rows) because a training step re-launches the same GEMMs.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}
// [rows, K] fp32, row stride ld elements, tile = box_rows x 32, SWIZZLE_128B (K-major operand tile)
static int tmap_2d(const float* base, int64_t rows, int64_t K, int64_t ld, int box_rows,
                   CUtensorMap* out) {
  using Key = std::tuple<const void*, int64_t, int64_t, int64_t, int>;
  static std::map<Key, CUtensorMap> cache;
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  const Key key{base, rows, K, ld, box_rows};
  auto it = cache.find(key);
  if (it != cache.end()) {
    *out = it->second;
    return B200RL_OK;
  }
  EncodeTiledFn fn = encode_tiled_fn();
  if (fn == nullptr) {
    set_error("tc2: cuTensorMapEncodeTiled is not available from this driver");
    return B200RL_ERR_UNSUPPORTED;
  }
  const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(float)};
  const cuuint32_t box[2] = {32u, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1u, 1u};
  CUtensorMap tm;
  CUresult r = fn(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides,
                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("tc2: cuTensorMapEncodeTiled failed (%d) for [%lld, %lld] ld %lld", (int)r,
              (long long)rows, (long long)K, (long long)ld);
    return B200RL_ERR_CUDA;
  }
  if (cache.size() > 4096) cache.clear();
  cache[key] = tm;
  *out = tm;
  return B200RL_OK;
}
template <class V>
static int tmap_for(const V&, int64_t, int64_t, int, CUtensorMap* out) {
  memset(out, 0, sizeof(*out));
  return B200RL_OK;
}
static int tmap_for(const ARow& v, int64_t rows, int64_t K, int box_rows, CUtensorMap* out) {
  return tmap_2d(v.p, rows, K, v.ld, box_rows, out);
}
static int tmap_for(const BCol& v, int64_t rows, int64_t K, int box_rows, CUtensorMap* out) {
  return tmap_2d(v.p, rows, K, v.ld, box_rows, out);
}

// operand base pointers (pair launches pass the second problem as byte offsets from the first)
static const void* view_base(const ARow& v) { return v.p; }
static const void* view_base(const ACol& v) { return v.p; }
static const void* view_base(const BRow& v) { return v.p; }
static const void* view_base(const BCol& v) { return v.p; }
static const void* view_base(const AConv<float>& v) { return v.v.x; }
static const void* view_base(const AConvT<float>& v) { return v.v.x; }
static const void* view_base(const AConvU8Raw& v) { return v.v.x; }
static const void* view_base(const AConvTU8Raw& v) { return v.v.x; }

// second problem of a pair launch (same shapes, see tc2::PairArgs)
template <class AL, class BL>
struct Tc2Pair {
  AL a;
  BL b;
  float* C;
  const float* bias;
};

template <int BN, int PASSES, int EPI, class AL, class BL>
static int launch_tc2_cfg(const AL& a, const BL& b, const GemmArgs& g, const tc2::EpiArgs& epi,
                          const Tc2Pair<AL, BL>* pair) {
  using L = tc2::Layout<BN, PASSES, AL::kExact>;
  auto kernel = tc2::tc2_gemm_kernel<BN, PASSES, EPI, AL, BL>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         L::kBytes);
    if (e != cudaSuccess) {
      set_error("tc2_gemm: cannot set dynamic smem to %d: %s", L::kBytes, cudaGetErrorString(e));
      return B200RL_ERR_CUDA;
    }
    configured = true;
  }
  tc2_env_flags();
  const int64_t tm1 = (g.M + tc2::kBM - 1) / tc2::kBM, tn = (g.N + BN - 1) / BN;
  const int64_t tm = pair ? 2 * tm1 : tm1;
  const int64_t tiles = tm * tn;
  int splits = 1;
  const int64_t target = kNumSMs;                  // one persistent CTA per SM
  if (tiles < target && g.K >= 8 * tc2::kBK && (g.ws != nullptr || EPI != tc2::EPI_STORE)) {
    int64_t want = target / tiles;
    int64_t max_by_k = g.K / (4 * tc2::kBK);
    int64_t max_by_ws = EPI != tc2::EPI_STORE ? 65535 : g.ws_bytes / (int64_t)((pair ? 2 : 1) * g.M * g.N * sizeof(float));
    int64_t s = want < max_by_k ? want : max_by_k;
    if (s > max_by_ws) s = max_by_ws;
    if (s >= 2) splits = (int)s;
  }
  int64_t kps = (g.K + splits - 1) / splits;
  kps = (kps + tc2::kBK - 1) / tc2::kBK * tc2::kBK;
  splits = (int)((g.K + kps - 1) / kps);
  if (splits < 1) splits = 1;
  const int64_t total = tiles * splits;
  B200RL_CHECK_ARG(total < (1ll << 31), "tc2_gemm: too many work items");
  const unsigned grid = (unsigned)(total < kNumSMs ? total : kNumSMs);
  CUtensorMap tmA, tmB, tmA2, tmB2;
  int rc = tmap_for(a, g.M, g.K, tc2::kBM, &tmA);
  if (rc) return rc;
  rc = tmap_for(b, g.N, g.K, BN, &tmB);
  if (rc) return rc;
  tmA2 = tmA;
  tmB2 = tmB;
  tc2::PairArgs pa{tm1, 0, 0, 0, 0};
  if (pair) {
    rc = tmap_for(pair->a, g.M, g.K, tc2::kBM, &tmA2);
    if (rc) return rc;
    rc = tmap_for(pair->b, g.N, g.K, BN, &tmB2);
    if (rc) return rc;
    pa.a_delta = (const char*)view_base(pair->a) - (const char*)view_base(a);
    pa.b_delta = (const char*)view_base(pair->b) - (const char*)view_base(b);
    pa.c_delta = pair->C - g.C;
    pa.bias_delta = (g.bias && pair->bias) ? pair->bias - g.bias : 0;
  }
  // epilogue-bound shapes (col2im scatter-add, short K loops) get all eight epilogue warps
  static const int epi_env = [] { const char* e = getenv("B200RL_TC2_EPI_WARPS"); return e ? atoi(e) : 0; }();
  const int epi_warps = (epi_env == 4 || epi_env == 8) ? epi_env
                        : (EPI == tc2::EPI_COL2IM || EPI == tc2::EPI_COL2IM_MERGE || kps <= 224) ? 8 : 4;
  // dynamic work distribution (b200rl_set_tile_scheduler) when a CTA has more than one item
  static int sched_seq = 0;
  int sched_slot = -1;
  if (total > grid && tile_scheduler_dynamic()) sched_slot = (sched_seq++) & (tc2::kSchedSlots - 1);
  B200RL_LAUNCH(kernel, grid, tc2::kThreads, L::kBytes, g.st, a, b, epi, g.C, g.bias, g.M, g.N, g.K, g.act, g.beta, splits, kps, (float*)g.ws, g.out_scale, tm, tn, epi_warps, sched_slot, pa, tmA, tmB, tmA2, tmB2);
  B200RL_CHECK_LAUNCH("tc2_gemm");
  if (splits > 1 && EPI == tc2::EPI_STORE) {
    const int64_t MN = g.M * g.N;
    B200RL_LAUNCH(splitk_reduce_kernel, (unsigned)((MN + 255) / 256), 256, 0, g.st, (const float*)g.ws, g.C, g.bias, MN, g.N, splits, g.act, g.beta, g.mask);
    B200RL_CHECK_LAUNCH("splitk_reduce");
    if (pair) {
      B200RL_LAUNCH(splitk_reduce_kernel, (unsigned)((MN + 255) / 256), 256, 0, g.st, (const float*)g.ws + (int64_t)splits * MN, pair->C, pair->bias, MN, g.N, splits, g.act, g.beta, g.mask);
      B200RL_CHECK_LAUNCH("splitk_reduce");
    }
  }
  return B200RL_OK;
}

// ---- one route rule for every dense / conv GEMM ------------------------------------------------
// Tensor route (tc2_gemm_kernel) when the GEMM mode allows it, the problem fills a tensor-core tile
// well enough, and both operand views can be moved as aligned 16-byte chunks; every other shape
// takes the fp32 FFMA kernel (launch_ffma).
template <class AL, class BL>
static bool tensor_route(const AL& a, const BL& b, const GemmArgs& g) {
  return gemm_mode() != 0 && g.N >= 16 && g.M >= 32 && g.K >= 8 && tc2_ok(a, g.M, g.K) &&
         tc2_ok(b, g.N, g.K);
}

// 3xTF32 in mode 1, 1xTF32 in mode 2.  BN by N; the col2im epilogues always use 128-column tiles
// (the merged one pairs columns 64 apart inside a tile).
template <int EPI, class AL, class BL>
static int launch_tensor(const AL& a, const BL& b, const GemmArgs& g, const tc2::EpiArgs& epi,
                         const Tc2Pair<AL, BL>* pair = nullptr) {
  constexpr bool kCol2im = EPI == tc2::EPI_COL2IM || EPI == tc2::EPI_COL2IM_MERGE;
  const bool one_pass = gemm_mode() == 2;
  if constexpr (!kCol2im) {
    if (g.N <= 32) return one_pass ? launch_tc2_cfg<32, 1, EPI>(a, b, g, epi, pair)
                                   : launch_tc2_cfg<32, 3, EPI>(a, b, g, epi, pair);
    if (g.N <= 64) return one_pass ? launch_tc2_cfg<64, 1, EPI>(a, b, g, epi, pair)
                                   : launch_tc2_cfg<64, 3, EPI>(a, b, g, epi, pair);
  }
  return one_pass ? launch_tc2_cfg<128, 1, EPI>(a, b, g, epi, pair)
                  : launch_tc2_cfg<128, 3, EPI>(a, b, g, epi, pair);
}

template <class AL, class BL>
static int launch_ffma(const AL& a, const BL& b, const GemmArgs& g) {
  if (g.N <= 32) return launch_gemm_cfg<128, 32, 4, 4>(a, b, g);
  if (g.N <= 64) {
    if (g.M >= 4096) return launch_gemm_cfg<128, 64, 8, 4>(a, b, g);
    return launch_gemm_cfg<64, 64, 4, 4>(a, b, g);
  }
  const int64_t t128 = ((g.M + 127) / 128) * ((g.N + 127) / 128);
  if (t128 >= kNumSMs) return launch_gemm_cfg<128, 128, 8, 8>(a, b, g);
  return launch_gemm_cfg<64, 64, 4, 4>(a, b, g);
}

// C = act(A @ B + bias) (* act'(mask)) (+ C when beta)
template <class AL, class BL>
static int launch_gemm(const AL& a, const BL& b, const GemmArgs& g) {
  if (g.M <= 0 || g.N <= 0) return B200RL_OK;
  B200RL_CHECK_ARG(g.K > 0, "gemm: K must be > 0");
  B200RL_CHECK_ARG(g.M < (1ll << 31) && g.N < (1ll << 31) && g.K < (1ll << 31), "gemm: dims");
  if (!tensor_route(a, b, g)) return launch_ffma(a, b, g);
  B200RL_CHECK_ARG(!(g.mask.y && g.beta), "gemm: an input-gradient mask cannot be combined with accumulation");
  tc2::EpiArgs epi{};
  epi.mask = g.mask;
  return launch_tensor<tc2::EPI_STORE>(a, b, g, epi);
}

// Weight-gradient GEMM (no bias / activation) on the tensor route: the split-K partials are
// accumulated with red.global.add straight into the (zeroed) gradient instead of going through a
// workspace + reduce kernel; summation order across splits is not fixed.  `db` (optional): bias
// gradient = column sums of B; for an MN-major B view they are accumulated by the converters of
// the same kernel and *db_fused is set, otherwise the caller runs the separate column-sum kernels.
template <class AL, class BL>
static int launch_grad_tensor(const AL& a, const BL& b, const GemmArgs& g, float* db, bool* db_fused) {
  const bool fuse_db = db != nullptr && !BL::kKContig && fuse_bias_grad();
  if (!g.beta) {
    cudaError_t e = cudaMemsetAsync(g.C, 0, (size_t)(g.M * g.N) * sizeof(float), g.st);
    if (e == cudaSuccess && fuse_db) e = cudaMemsetAsync(db, 0, (size_t)g.N * sizeof(float), g.st);
    if (e != cudaSuccess) {
      set_error("grad gemm: memset failed: %s", cudaGetErrorString(e));
      return B200RL_ERR_CUDA;
    }
  }
  tc2::EpiArgs epi{};
  if (fuse_db) epi.colsum = db;
  *db_fused = fuse_db;
  return launch_tensor<tc2::EPI_ATOMIC>(a, b, g, epi);
}
template <class AL, class BL>
static int launch_grad_gemm(const AL& a, const BL& b, const GemmArgs& g, float* db, bool* db_fused) {
  *db_fused = false;
  if (!tensor_route(a, b, g)) return launch_gemm(a, b, g);   // FFMA route
  return launch_grad_tensor(a, b, g, db, db_fused);
}

// ---- skinny-head dispatch (N <= 16) ----------------------------------------------------------
static bool skinny_ok(int64_t M, int64_t K, int64_t N) {
  return gemm_mode() != 0 && skinny_enabled() && N >= 1 && N <= kSkinnyMaxN && K >= 1 && K <= 1024 &&
         K * N * (int64_t)sizeof(float) <= kSkinnySmem && M >= 1;
}
template <int NMAX>
static int skinny_fwd_launch(const float* X, int64_t ldx, const float* W, const float* bias,
                             float* Y, int64_t M, int64_t K, int64_t N, int act, cudaStream_t st) {
  int64_t blocks = (M + 7) / 8;
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  B200RL_LAUNCH(skinny_fwd_kernel<NMAX>, (unsigned)blocks, 256, (size_t)(K * N * sizeof(float)), st, X, ldx, W, bias, Y, M, (int)K, (int)N, act);
  B200RL_CHECK_LAUNCH("skinny_fwd");
  return B200RL_OK;
}
template <int NMAX>
static int skinny_dx_launch(const float* dY, const float* W, float* dX, int64_t M, int64_t K,
                            int64_t N, const ActMask& mask, cudaStream_t st) {
  int64_t blocks = (M * ((K + 3) / 4) + 255) / 256;
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  B200RL_LAUNCH(skinny_dx_kernel<NMAX>, (unsigned)blocks, 256, (size_t)(K * N * sizeof(float)), st, dY, W, dX, M, (int)K, (int)N, mask);
  B200RL_CHECK_LAUNCH("skinny_dx");
  return B200RL_OK;
}
template <int NMAX>
static int skinny_dw_launch(const float* X, int64_t ldx, const float* dY, float* dW, float* db,
                            int64_t M, int64_t K, int64_t N, int accumulate, cudaStream_t st) {
  if (!accumulate) {
    cudaError_t e = cudaMemsetAsync(dW, 0, (size_t)(K * N) * sizeof(float), st);
    if (e == cudaSuccess && db) e = cudaMemsetAsync(db, 0, (size_t)N * sizeof(float), st);
    if (e != cudaSuccess) {
      set_error("skinny dW: memset failed: %s", cudaGetErrorString(e));
      return B200RL_ERR_CUDA;
    }
  }
  int64_t rows = (M + 2 * kNumSMs - 1) / (2 * kNumSMs);   // ~2 CTAs per SM; small M: 8-row slabs
  rows = (rows + 7) / 8 * 8;
  const int64_t blocks = (M + rows - 1) / rows;
  if (K <= 256) B200RL_LAUNCH((skinny_dw_kernel<NMAX, 1>), (unsigned)blocks, 256, (size_t)(K * N * sizeof(float)), st, X, ldx, dY, dW, db, M, (int)K, (int)N, rows);
  else if (K <= 512) B200RL_LAUNCH((skinny_dw_kernel<NMAX, 2>), (unsigned)blocks, 256, 0, st, X, ldx, dY, dW, db, M, (int)K, (int)N, rows);
  else B200RL_LAUNCH((skinny_dw_kernel<NMAX, 4>), (unsigned)blocks, 256, 0, st, X, ldx, dY, dW, db, M, (int)K, (int)N, rows);
  B200RL_CHECK_LAUNCH("skinny_dw");
  return B200RL_OK;
}
#define SKINNY_BY_N(fn, N, ...)                                  \
  ((N) <= 4 ? fn<4>(__VA_ARGS__) : (N) <= 8 ? fn<8>(__VA_ARGS__) : fn<16>(__VA_ARGS__))

static int colsum(const float* dZ, float* db, int64_t M, int64_t N, int beta, void* ws,
                  int64_t ws_bytes, cudaStream_t st) {
  const int64_t nparts = (M + kColRows - 1) / kColRows;
  B200RL_CHECK_ARG(ws != nullptr && ws_bytes >= (int64_t)(nparts * N * sizeof(float)),
                   "bias gradient needs %lld bytes of workspace",
                   (long long)(nparts * N * sizeof(float)));
  B200RL_CHECK_ARG(nparts <= 65535, "bias gradient: too many rows");
  dim3 grid((unsigned)((N + 31) / 32), (unsigned)nparts);
  B200RL_LAUNCH(colsum_partial_kernel, grid, 256, 0, st, dZ, (float*)ws, M, N);
  B200RL_CHECK_LAUNCH("colsum_partial");
  B200RL_LAUNCH(colsum_final_kernel, (unsigned)((N + 7) / 8), 256, 0, st, (const float*)ws, db, nparts, N, beta);
  B200RL_CHECK_LAUNCH("colsum_final");
  return B200RL_OK;
}

static int make_geom(const b200rl_conv_t* c, ConvGeom& g) {
  B200RL_CHECK_ARG(c != nullptr, "conv geometry is NULL");
  B200RL_CHECK_ARG(c->N > 0 && c->H > 0 && c->W > 0 && c->C > 0 && c->KH > 0 && c->KW > 0 &&
                       c->F > 0 && c->stride > 0,
                   "conv: non-positive dimension");
  B200RL_CHECK_ARG(c->H >= c->KH && c->W >= c->KW, "conv: kernel larger than input");
  g.H = c->H; g.W = c->W; g.C = c->C; g.KH = c->KH; g.KW = c->KW; g.F = c->F;
  g.stride = c->stride;
  g.OH = (c->H - c->KH) / c->stride + 1;
  g.OW = (c->W - c->KW) / c->stride + 1;
  g.d_ohow = FastDiv((uint32_t)(g.OH * g.OW));
  g.d_ow = FastDiv((uint32_t)g.OW);
  g.d_kwc = FastDiv((uint32_t)(g.KW * g.C));
  g.in_row = (int64_t)c->W * c->C;
  g.in_img = c->x_batch_stride > 0 ? c->x_batch_stride : (int64_t)c->H * c->W * c->C;
  const int64_t M = (int64_t)c->N * g.OH * g.OW;
  B200RL_CHECK_ARG(M < (1ll << 31), "conv: too many output positions");
  return B200RL_OK;
}

}  // namespace b200rl

using namespace b200rl;

// Forward pass of TWO layers of identical shape in one launch (DQN: the online network on
// obs[:, 0] and the target network on obs[:, T-1]): when both problems take the tensor route and
// both or neither have a bias.  Otherwise the callers make two single calls.
static int pair_fwd_enabled() {
  static const int v = [] { const char* e = getenv("B200RL_PAIR_FWD"); return e ? atoi(e) : 1; }();
  return v;
}
template <class AL, class BL>
static bool pair_route(const AL& a1, const BL& b1, const GemmArgs& g1, const AL& a2, const BL& b2,
                       const GemmArgs& g2) {
  return pair_fwd_enabled() && tensor_route(a1, b1, g1) && tensor_route(a2, b2, g2) &&
         (g1.bias == nullptr) == (g2.bias == nullptr);
}
template <class AL, class BL>
static int launch_pair(const AL& a1, const BL& b1, const GemmArgs& g1, const AL& a2, const BL& b2,
                       const GemmArgs& g2) {
  const Tc2Pair<AL, BL> p{a2, b2, g2.C, g2.bias};
  return launch_tensor<tc2::EPI_STORE>(a1, b1, g1, tc2::EpiArgs{}, &p);
}


extern "C" {

int b200rl_tc2_trace_buffer(long long* dev_buf) {
  cudaError_t e = cudaMemcpyToSymbol(tc2::g_tc2_trace, &dev_buf, sizeof(dev_buf));
  if (e != cudaSuccess) {
    set_error("tc2_trace_buffer: %s", cudaGetErrorString(e));
    return B200RL_ERR_CUDA;
  }
  return B200RL_OK;
}

int b200rl_set_tile_scheduler(int dynamic) {
  g_tile_sched = dynamic ? 1 : 0;
  return B200RL_OK;
}

int b200rl_set_tc2_flags(int flags) {
  cudaError_t e = cudaMemcpyToSymbol(tc2::g_tc2_flags, &flags, sizeof(flags));
  if (e != cudaSuccess) {
    set_error("set_tc2_flags: %s", cudaGetErrorString(e));
    return B200RL_ERR_CUDA;
  }
  return B200RL_OK;
}

// ---- thin-input dispatch (K <= 32, 16 < N <= 256, N % 4 == 0) -----------------------------------
static bool thin_ok(const float* X, int64_t ldx, const float* W, int64_t M, int64_t K, int64_t N) {
  return gemm_mode() != 0 && thin_enabled() && K >= 1 && K <= kThinMaxK && N > kSkinnyMaxN &&
         N <= kThinMaxN && (N & 3) == 0 && M >= 1 && al16(W);
}
static int thin_fwd_launch(const float* X, int64_t ldx, const float* W, const float* bias, float* Y,
                           int64_t M, int64_t K, int64_t N, int act, cudaStream_t st) {
  const int64_t chunks = (M + kThinRows - 1) / kThinRows;
  const int KP = ((int)K + 3) & ~3;
  const size_t smem = (size_t)KP * N * sizeof(float) + (size_t)kThinRows * KP * sizeof(float);
  const int64_t blocks = chunks < 4 * kNumSMs ? chunks : 4 * kNumSMs;
  B200RL_LAUNCH(thin_fwd_kernel, (unsigned)blocks, 256, smem, st, X, ldx, W, bias, Y, M, (int)K, (int)N, act, chunks);
  B200RL_CHECK_LAUNCH("thin_fwd");
  return B200RL_OK;
}
static int thin_dw_launch(const float* X, int64_t ldx, const float* dZ, float* dW, float* db,
                          int64_t M, int64_t K, int64_t N, int accumulate, cudaStream_t st) {
  if (!accumulate) {
    cudaError_t e = cudaMemsetAsync(dW, 0, (size_t)(K * N) * sizeof(float), st);
    if (e == cudaSuccess && db) e = cudaMemsetAsync(db, 0, (size_t)N * sizeof(float), st);
    if (e != cudaSuccess) {
      set_error("thin dW: memset failed: %s", cudaGetErrorString(e));
      return B200RL_ERR_CUDA;
    }
  }
  int64_t rows = (M + 4 * kNumSMs - 1) / (4 * kNumSMs);
  rows = (rows + kThinRows - 1) / kThinRows * kThinRows;
  const int64_t blocks = (M + rows - 1) / rows;
  const int KMAX = K <= 8 ? 8 : K <= 20 ? 20 : 32;
  const size_t smem = ((size_t)kThinRows * KMAX + (size_t)(K + 1) * N) * sizeof(float);
  if (KMAX == 8) B200RL_LAUNCH(thin_dw_kernel<8>, (unsigned)blocks, 256, smem, st, X, ldx, dZ, dW, db, M, (int)K, (int)N, rows);
  else if (KMAX == 20) B200RL_LAUNCH(thin_dw_kernel<20>, (unsigned)blocks, 256, smem, st, X, ldx, dZ, dW, db, M, (int)K, (int)N, rows);
  else B200RL_LAUNCH(thin_dw_kernel<32>, (unsigned)blocks, 256, smem, st, X, ldx, dZ, dW, db, M, (int)K, (int)N, rows);
  B200RL_CHECK_LAUNCH("thin_dw");
  return B200RL_OK;
}

int b200rl_set_gemm_mode(int mode) {
  B200RL_CHECK_ARG(mode >= 0 && mode <= 2, "gemm mode must be 0 (fp32 FFMA), 1 (tcgen05 3xTF32) "
                                           "or 2 (tcgen05 1xTF32)");
  g_gemm_mode = mode;
  return B200RL_OK;
}

int b200rl_dense_fwd(const float* X, int64_t ldx, const float* W, const float* bias, float* Y,
                     int64_t M, int64_t K, int64_t N, int act, void* workspace,
                     int64_t ws_bytes, void* stream) {
  B200RL_CHECK_ARG(X && W && Y, "dense_fwd: NULL argument");
  B200RL_CHECK_ARG(ldx == 0 || ldx >= K, "dense_fwd: ldx < K");
  if (skinny_ok(M, K, N))
    return SKINNY_BY_N(skinny_fwd_launch, N, X, ldx ? ldx : K, W, bias, Y, M, K, N, act,
                       (cudaStream_t)stream);
  if (thin_ok(X, ldx, W, M, K, N) && al16(Y) && (bias == nullptr || al16(bias)))
    return thin_fwd_launch(X, ldx ? ldx : K, W, bias, Y, M, K, N, act, (cudaStream_t)stream);
  GemmArgs g{Y, bias, M, N, K, act, 0, workspace, ws_bytes, (cudaStream_t)stream};
  return launch_gemm(ARow{X, ldx ? ldx : K}, BRow{W, N}, g);
}

int b200rl_dense_fwd_pair(const float* X1, const float* X2, int64_t ldx, const float* W1,
                          const float* W2, const float* bias1, const float* bias2, float* Y1,
                          float* Y2, int64_t M, int64_t K, int64_t N, int act, void* workspace,
                          int64_t ws_bytes, void* stream) {
  B200RL_CHECK_ARG(X1 && X2 && W1 && W2 && Y1 && Y2, "dense_fwd_pair: NULL argument");
  B200RL_CHECK_ARG(ldx == 0 || ldx >= K, "dense_fwd_pair: ldx < K");
  if (skinny_ok(M, K, N) || (thin_ok(X1, ldx, W1, M, K, N) && thin_ok(X2, ldx, W2, M, K, N))) {
    int rc = b200rl_dense_fwd(X1, ldx, W1, bias1, Y1, M, K, N, act, workspace, ws_bytes, stream);
    if (rc) return rc;
    return b200rl_dense_fwd(X2, ldx, W2, bias2, Y2, M, K, N, act, workspace, ws_bytes, stream);
  }
  const GemmArgs g1{Y1, bias1, M, N, K, act, 0, workspace, ws_bytes, (cudaStream_t)stream};
  const GemmArgs g2{Y2, bias2, M, N, K, act, 0, workspace, ws_bytes, (cudaStream_t)stream};
  const ARow a1{X1, ldx ? ldx : K}, a2{X2, ldx ? ldx : K};
  const BRow b1{W1, N}, b2{W2, N};
  if (pair_route(a1, b1, g1, a2, b2, g2)) return launch_pair(a1, b1, g1, a2, b2, g2);
  int rc = launch_gemm(a1, b1, g1);
  if (rc) return rc;
  return launch_gemm(a2, b2, g2);
}

int b200rl_dense_bwd(const float* X, int64_t ldx, const float* W, const float* dY, float* dX,
                     float* dW, float* db, int64_t M, int64_t K, int64_t N, int accumulate,
                     int x_act, void* workspace, int64_t ws_bytes, void* stream) {
  B200RL_CHECK_ARG(X && W && dY, "dense_bwd: NULL argument");
  B200RL_CHECK_ARG(ldx == 0 || ldx >= K, "dense_bwd: ldx < K");
  B200RL_CHECK_ARG(x_act >= B200RL_ACT_NONE && x_act <= B200RL_ACT_TANH, "dense_bwd: x_act");
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  if (skinny_ok(M, K, N)) {
    if (dX) {
      ActMask mask{};
      if (x_act != B200RL_ACT_NONE) mask = ActMask{X, ldx ? ldx : K, x_act};
      rc = SKINNY_BY_N(skinny_dx_launch, N, dY, W, dX, M, K, N, mask, st);
      if (rc) return rc;
    }
    if (dW) {
      rc = SKINNY_BY_N(skinny_dw_launch, N, X, ldx ? ldx : K, dY, dW, db, M, K, N, accumulate, st);
      if (rc) return rc;
    } else if (db) {
      rc = colsum(dY, db, M, N, accumulate, workspace, ws_bytes, st);
      if (rc) return rc;
    }
    return B200RL_OK;
  }
  if (dX) {
    GemmArgs g{dX, nullptr, M, K, N, B200RL_ACT_NONE, 0, workspace, ws_bytes, st};
    if (x_act != B200RL_ACT_NONE) g.mask = ActMask{X, ldx ? ldx : K, x_act};
    rc = launch_gemm(ARow{dY, N}, BCol{W, N}, g);
    if (rc) return rc;
  }
  bool db_fused = false;
  if (dW && thin_ok(X, ldx, W, M, K, N) && al16(dY)) {
    rc = thin_dw_launch(X, ldx ? ldx : K, dY, dW, db, M, K, N, accumulate, st);
    if (rc) return rc;
    db_fused = true;
  } else if (dW) {
    GemmArgs g{dW, nullptr, K, N, M, B200RL_ACT_NONE, accumulate, workspace, ws_bytes, st};
    rc = launch_grad_gemm(ACol{X, ldx ? ldx : K}, BRow{dY, N}, g, db, &db_fused);
    if (rc) return rc;
  }
  if (db && !db_fused) {
    rc = colsum(dY, db, M, N, accumulate, workspace, ws_bytes, st);
    if (rc) return rc;
  }
  return B200RL_OK;
}

int b200rl_act_bwd(const float* Y, const float* dY, float* dZ, int64_t n, int act,
                   void* stream) {
  B200RL_CHECK_ARG(Y && dY && dZ && n >= 0, "act_bwd: bad argument");
  if (n == 0) return B200RL_OK;
  const int vec = (n & 3) == 0 && ((((uintptr_t)Y | (uintptr_t)dY | (uintptr_t)dZ) & 15) == 0);
  int64_t blocks = ((vec ? n / 4 : n) + 255) / 256;
  if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
  B200RL_LAUNCH(act_bwd_kernel, (unsigned)blocks, 256, 0, (cudaStream_t)stream, Y, dY, dZ, n, act, vec);
  B200RL_CHECK_LAUNCH("act_bwd");
  return B200RL_OK;
}

int b200rl_conv2d_fwd(const void* X, int x_is_u8, float x_scale, const float* Wt,
                      const float* bias, float* Y, const b200rl_conv_t* c, int act,
                      void* workspace, int64_t ws_bytes, void* stream) {
  B200RL_CHECK_ARG(X && Wt && Y, "conv2d_fwd: NULL argument");
  ConvGeom cg;
  int rc = make_geom(c, cg);
  if (rc) return rc;
  const int64_t M = (int64_t)c->N * cg.OH * cg.OW, K = (int64_t)c->KH * c->KW * c->C;
  GemmArgs g{Y, bias, M, c->F, K, act, 0, workspace, ws_bytes, (cudaStream_t)stream};
  const BRow w{Wt, c->F};
  if (x_is_u8) {
    // raw pixels on the tensor route (1/x_scale applied to the accumulator), the reference's exact
    // cast and division on the FFMA route
    const ConvView<uint8_t> v{(const uint8_t*)X, cg, x_scale};
    if (!tensor_route(AConvU8Raw{v}, w, g)) return launch_ffma(AConv<uint8_t>{v}, w, g);
    g.out_scale = 1.f / x_scale;
    return launch_tensor<tc2::EPI_STORE>(AConvU8Raw{v}, w, g, tc2::EpiArgs{});
  }
  return launch_gemm(AConv<float>{ConvView<float>{(const float*)X, cg, 1.f}}, w, g);
}

int b200rl_conv2d_fwd_pair(const void* X1, const void* X2, int x_is_u8, float x_scale,
                           const float* Wt1, const float* Wt2, const float* bias1,
                           const float* bias2, float* Y1, float* Y2, const b200rl_conv_t* c,
                           int act, void* workspace, int64_t ws_bytes, void* stream) {
  B200RL_CHECK_ARG(X1 && X2 && Wt1 && Wt2 && Y1 && Y2, "conv2d_fwd_pair: NULL argument");
  ConvGeom cg;
  int rc = make_geom(c, cg);
  if (rc) return rc;
  const int64_t M = (int64_t)c->N * cg.OH * cg.OW, K = (int64_t)c->KH * c->KW * c->C;
  GemmArgs g1{Y1, bias1, M, c->F, K, act, 0, workspace, ws_bytes, (cudaStream_t)stream};
  const GemmArgs g2{Y2, bias2, M, c->F, K, act, 0, workspace, ws_bytes, (cudaStream_t)stream};
  const BRow b1{Wt1, c->F}, b2{Wt2, c->F};
  if (x_is_u8) {
    const AConvU8Raw a1{ConvView<uint8_t>{(const uint8_t*)X1, cg, x_scale}};
    const AConvU8Raw a2{ConvView<uint8_t>{(const uint8_t*)X2, cg, x_scale}};
    if (pair_route(a1, b1, g1, a2, b2, g2)) {
      g1.out_scale = 1.f / x_scale;
      return launch_pair(a1, b1, g1, a2, b2, g2);
    }
  } else {
    const AConv<float> a1{ConvView<float>{(const float*)X1, cg, 1.f}};
    const AConv<float> a2{ConvView<float>{(const float*)X2, cg, 1.f}};
    if (pair_route(a1, b1, g1, a2, b2, g2)) return launch_pair(a1, b1, g1, a2, b2, g2);
  }
  rc = b200rl_conv2d_fwd(X1, x_is_u8, x_scale, Wt1, bias1, Y1, c, act, workspace, ws_bytes, stream);
  if (rc) return rc;
  return b200rl_conv2d_fwd(X2, x_is_u8, x_scale, Wt2, bias2, Y2, c, act, workspace, ws_bytes, stream);
}

int b200rl_conv2d_bwd(const void* X, int x_is_u8, float x_scale, const float* Wt,
                      const float* dY, float* dX, float* dW, float* db,
                      const b200rl_conv_t* c, int accumulate, int x_act, void* workspace,
                      int64_t ws_bytes, void* stream) {
  B200RL_CHECK_ARG(X && Wt && dY, "conv2d_bwd: NULL argument");
  B200RL_CHECK_ARG(!(dX && x_is_u8), "conv2d_bwd: no input gradient for u8 input");
  B200RL_CHECK_ARG(x_act >= B200RL_ACT_NONE && x_act <= B200RL_ACT_TANH, "conv2d_bwd: x_act");
  ConvGeom cg;
  int rc = make_geom(c, cg);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t M = (int64_t)c->N * cg.OH * cg.OW, K = (int64_t)c->KH * c->KW * c->C;
  const int64_t F = c->F;
  ActMask mask{};
  if (x_act != B200RL_ACT_NONE && !x_is_u8) mask = ActMask{(const float*)X, cg.in_img, x_act};
  bool db_fused = false;
  if (dW) {  // dW[K,F] = im2col(X)^T @ dY
    GemmArgs g{dW, nullptr, K, F, M, B200RL_ACT_NONE, accumulate, workspace, ws_bytes, st};
    const BRow dy{dY, F};
    if (x_is_u8) {   // the two views of b200rl_conv2d_fwd
      const ConvView<uint8_t> v{(const uint8_t*)X, cg, x_scale};
      if (tensor_route(AConvTU8Raw{v}, dy, g)) {
        g.out_scale = 1.f / x_scale;
        rc = launch_grad_tensor(AConvTU8Raw{v}, dy, g, db, &db_fused);
      } else {
        rc = launch_ffma(AConvT<uint8_t>{v}, dy, g);
      }
    } else {
      rc = launch_grad_gemm(AConvT<float>{ConvView<float>{(const float*)X, cg, 1.f}}, dy, g, db, &db_fused);
    }
    if (rc) return rc;
  }
  if (db && !db_fused) {
    rc = colsum(dY, db, M, F, accumulate, workspace, ws_bytes, st);
    if (rc) return rc;
  }
  if (!dX) return B200RL_OK;
  const int64_t total = (int64_t)c->N * c->H * c->W * c->C;
  const ARow da{dY, F};
  const BCol wt{Wt, F};
  GemmArgs g{nullptr, nullptr, M, K, F, B200RL_ACT_NONE, 0, nullptr, 0, st};
  if ((c->C & 3) == 0 && tensor_route(da, wt, g)) {
    // dY @ W^T with the col2im scatter-add fused into the epilogue
    cudaError_t e = cudaMemsetAsync(dX, 0, (size_t)total * sizeof(float), st);
    if (e != cudaSuccess) {
      set_error("conv2d_bwd: memset failed: %s", cudaGetErrorString(e));
      return B200RL_ERR_CUDA;
    }
    tc2::EpiArgs epi{cg, dX};
    epi.mask = mask;
    // neighbour pre-sum of the col2im epilogue (tc2_gemm.cuh): the partner column group sits
    // stride * C = 64 columns away, i.e. in the other half of the same 128-column tile (the Mnih
    // conv2 (k4 s2 C32) and conv3 (k3 s1 C64) input gradients); B200RL_COL2IM_MERGE=0 turns it off
    static const int merge_env = [] { const char* e = getenv("B200RL_COL2IM_MERGE"); return e ? atoi(e) : 1; }();
    if (merge_env && (int64_t)c->stride * c->C == 64 && (c->C & 15) == 0 && cg.OW > 1) {
      epi.merge_cols = 64;
      return launch_tensor<tc2::EPI_COL2IM_MERGE>(da, wt, g, epi);
    }
    return launch_tensor<tc2::EPI_COL2IM>(da, wt, g, epi);
  }
  // dcol[M,K] = dY @ W^T, then gather-form col2im
  const int64_t need = M * K * (int64_t)sizeof(float);
  B200RL_CHECK_ARG(workspace && ws_bytes >= need,
                   "conv2d_bwd: input gradient needs %lld bytes of workspace", (long long)need);
  g.C = (float*)workspace;
  rc = launch_gemm(da, wt, g);
  if (rc) return rc;
  B200RL_LAUNCH(col2im_kernel, (unsigned)((total + 255) / 256), 256, 0, st, (const float*)workspace, dX, cg, total, (int)K, mask);
  B200RL_CHECK_LAUNCH("col2im");
  return B200RL_OK;
}

}  // extern "C"
