// Persistent, warp-specialised tcgen05 GEMM for the Q / actor / critic networks: tcgen05.mma
// (kind::tf32) with TMEM accumulators, fp32-grade accuracy through the 3xTF32 split.
//
//   C[M,N] (+)= act(A[M,K] @ B[K,N] + bias)   over the operand views of nn.cu, 3xTF32 or 1xTF32
//
// Why 3xTF32: north_star parity is 1e-5 relative on the loss; one TF32 pass keeps ~11 mantissa
// bits (1e-3).  Each fp32 operand x is split into hi = x with the low 13 mantissa bits cleared and
// lo = x - hi (exact); the tensor core accumulates lo_a*hi_b + hi_a*lo_b + hi_a*hi_b into the same
// fp32 TMEM accumulator (the dropped lo*lo term is 2^-22 relative).  Raw uint8 pixels are exact in
// TF32, so an exact A operand needs no lo plane (a*b_lo + a*b_hi).
//
// History (profiles/r2/README.md, run 1): the first-generation kernel ran ONE output tile per CTA
// with 8 producer warps that pulled operands through registers (LDG -> split -> STS); ncu showed
// (a) 80-225 KB of SASS per instantiation, i.e. an instruction cache that never warms, (b)
// producers stalled on their own loads, (c) the prologue (TMEM allocation, barrier init) and the
// epilogue exposed on every tile.  Here:
//
//   * one CTA per SM, persistent over (split, m-tile, n-tile) work items;
//   * warps 0-7   LOADERS: cp.async (LDGSTS, 16 B, zero-fill) of the raw operand chunks straight
//                 into their final 128B-swizzled position of a deep stage ring; completion is
//                 signalled with cp.async.mbarrier.arrive.noinc, so the loader never waits for
//                 data and runs ahead by the full ring; plain row-major 2-D operands are one
//                 cp.async.bulk.tensor (TMA) per tile instead;
//   * warps 8-15  CONVERTERS: shared -> shared; compute the TF32 lo plane of every fp32 chunk
//                 (the raw tile is the hi plane), or expand raw uint8 pixels to fp32; linear,
//                 conflict-free addressing, no global address arithmetic; they also accumulate
//                 the fused bias gradient (column sums of B) of weight-gradient GEMMs;
//   * warp 16     one thread issues tcgen05.mma into one of TWO TMEM accumulators; the hi and lo
//                 planes of B form one operand of N = 2 BN columns (Layout::kWide), so a 3xTF32
//                 K step is 2 MMAs and an exact-A (uint8) step is 1;
//   * warps 17+   EPILOGUE of tile i (tcgen05.ld, bias/activation/act' mask, stores, split-K
//                 red.add, fused col2im scatter-add) overlaps the main loop of tile i+1;
//   * every loop that is not a fixed 4-8x unroll is rolled.  There are no scalar paths: the host
//                 dispatch only sends views whose every 16-byte chunk is contiguous and aligned
//                 (tc2_ok in nn.cu); every other shape takes the FFMA kernel.
//
// Descriptors follow cute/arch/mma_sm100_desc.hpp (SmemDescriptor: K-major SWIZZLE_128B,
// SBO = 1024 B, version 1; InstrDescriptor: F32 accumulate, TF32 x TF32, M = 128, N = BN).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

namespace b200rl {
namespace tc2 {

// ---- tcgen05 / mbarrier primitives, shared-memory layouts ---------------------------------------
constexpr int kBM = 128;
constexpr int kBK = 32;                    // fp32 elements = 128 bytes = one swizzle row

__device__ __forceinline__ uint32_t smem_addr(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Spin on the non-blocking test_wait (the `poll` A/B switch, bit 6 of g_tc2_flags; the default
// is the suspending try_wait of mbar_wait_hw below).
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// K-major, SWIZZLE_128B, 8-row groups 1024 B apart (cute SmemDescriptor, version 1).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);          // start address
  d |= (uint64_t)1 << 16;                          // leading byte offset (unused for SW128 K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                // stride byte offset
  d |= (uint64_t)1 << 46;                          // version = 1 (sm_100)
  d |= (uint64_t)2 << 61;                          // layout type SWIZZLE_128B
  return d;
}
// MN-major tf32 operands: SWIZZLE_128B_BASE32B is the only layout the tensor core accepts for
// 32-bit MN-major data (cutlass sm100_common.inl: "for mn-major tf32 operands, SW128_32B is the
// only available smem layout"; cute Layout_MN_SW128_32B_Atom = Swizzle<2,5,2> o (1024 bit, 4) :
// (1, 1024 bit)).  A k-row holds 32 consecutive M/N elements (128 B); 4 k-rows form a 512 B atom
// in which the 32-byte blocks of a row are XORed with the row index; LBO = distance between
// 32-element M/N groups, SBO = distance between 4-row k atoms (one K=8 MMA spans two atoms).
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t saddr, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)(512 >> 4) << 16;                 // LBO: next 32-row M/N group (adjacent atom)
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;  // SBO: next 4-row k atom = (ROWS/32) atoms
  d |= (uint64_t)1 << 46;                          // version = 1 (sm_100)
  d |= (uint64_t)1 << 61;                          // layout type 1 = SWIZZLE_128B_BASE32B
  return d;
}
__host__ __device__ constexpr uint32_t make_idesc(int bn, bool a_mn, bool b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
}
// byte offset of the 16-byte chunk holding rows 4*cm..4*cm+3 at reduction index k (0..31) in an
// MN-major tile: 512 B atoms (32 rows x 4 k) tiled M/N-fastest (the arrangement cute's
// tile_to_shape produces), rows 128 B apart; inside a row the 32-byte block index is XORed with
// (k & 3).
template <int ROWS>
__device__ __forceinline__ uint32_t mn128(uint32_t cm, uint32_t k) {
  const uint32_t c = cm & 7u, kin = k & 3u;
  const uint32_t blk = (((c >> 1) ^ kin) << 1) | (c & 1u);   // 32-byte block XOR k, 16 B half kept
  return ((k >> 2) * (ROWS / 32) + (cm >> 3)) * 512u + kin * 128u + (blk << 4);
}
// byte offset of 16-byte chunk j (0..7) of row r inside a K-major [rows x 128 B] SWIZZLE_128B tile
__device__ __forceinline__ uint32_t sw128(uint32_t r, uint32_t j) {
  return (r >> 3) * 1024u + (r & 7u) * 128u + ((j ^ (r & 7u)) << 4);
}

// Epilogue variants.  EPI_STORE: C (+)= act(acc + bias) or split-K partial.  EPI_ATOMIC: C += acc
// with red.global.add (split-K without a reduce pass; C pre-zeroed).  EPI_COL2IM: the GEMM is
// dcol[pos, (ky,kx,c)] = dY @ W^T of a convolution input gradient and every 4-channel group is
// scatter-added straight into dX[n, oy*s+ky, ox*s+kx, c..c+3] with one red.global.add.v4.f32 --
// the [M, KH*KW*C] dcol matrix is never materialised and split-K partials need no reduction pass
// (dX must be zeroed by the caller; summation order of the <= KH*KW/s^2 contributions per element
// is not fixed).  EPI_COL2IM_MERGE: EPI_COL2IM with the neighbour pre-sum of EpiArgs::merge_cols
// (its own instantiation, so that neither variant pays for the other's registers).
constexpr int EPI_STORE = 0;
constexpr int EPI_COL2IM = 1;
constexpr int EPI_ATOMIC = 2;
constexpr int EPI_COL2IM_MERGE = 3;
struct EpiArgs {
  ConvGeom g;
  float* dx;
  ActMask mask;     // EPI_STORE / EPI_COL2IM: multiply the input gradient by act'(mask.y)
  float* colsum;    // EPI_ATOMIC with an MN-major B view: column sums of B (bias gradient) += here
  // EPI_COL2IM_MERGE: columns c and c + merge_cols (= stride * C) of NEIGHBOURING output positions
  // (ox + 1, ox) address the same input element; the epilogue adds them with a lane shuffle before
  // the red.global.add.  0: every column group is scattered.
  int merge_cols;
};

// ---- the persistent kernel ----------------------------------------------------------------------
// Run-7 trace: once the MMA count per K step dropped (WIDE below), the K-block period (620-720 ns)
// stayed above every role's busy time (loaders ~400-500, converters ~350-450, MMA issue ~230-410):
// a loader and a converter warp share each scheduler and both are chains of dependent scalar
// instructions (address arithmetic -> LDGSTS; LDS -> split -> STS), i.e. latency- not
// throughput-bound.  Two warps per role per scheduler hide that latency.
constexpr int kLoaderThreads = 256;
constexpr int kConvThreads = 256;
constexpr int kMmaWarp = (kLoaderThreads + kConvThreads) / 32;
constexpr int kFirstEpiWarp = kMmaWarp + 1;
// Epilogue warps: 8 are launched; `epi_warps` (4 or 8, per launch) of them work, the others park
// on the closing barrier.  Run 8: with 8 working warps (two per TMEM lane quadrant, each draining
// half of the columns) the epilogue-bound GEMMs (col2im scatter, K <= ~200) are 5-35 % faster,
// the main-loop-bound ones 2-5 % slower (eight more warps polling accumulator barriers).
constexpr int kEpiWarps = 8;
constexpr int kThreads = (kFirstEpiWarp + kEpiWarps) * 32;
static_assert(kLoaderThreads == 256 && kConvThreads == 256, "thread -> chunk maps below assume 256");

// The tensor core ignores the low 13 mantissa bits of a TF32 operand, so the raw fp32 tile IS the
// hi plane and only the lo plane is computed (x - (x & 0xFFFFE000)); measured bit-identical to
// the explicitly masked hi plane on every layer (profiles/r2/run2_tc2_check*.jsonl).
// bit 0 of the flags: store the masked hi plane anyway (A/B switch for tests/profiles).
// bits 3/4/5: ABLATIONS for profiles/tc2_ablate.py (results are garbage, only the time is read):
// loaders issue no copies / converters do no work / the MMA thread issues no MMAs.
__device__ int g_tc2_flags = 0;
// optional pipeline trace (b200rl_tc2_trace_buffer): CTA 0 stamps %globaltimer at the start and end
// of every pipeline step of each role: trace[role][step][2], role 0 loader / 1 converter / 2 MMA /
// 3 epilogue (steps are K blocks for roles 0-2 and tiles for role 3), first kTraceSteps steps.
// Dynamic tile scheduler: {next work item, finished CTAs} per launch, taken round-robin from this
// pool by the host (concurrent launches of one stream fork use different slots); a launch leaves
// its slot zeroed.  sched_slot < 0: static striding (blockIdx.x + i * gridDim.x).
constexpr int kSchedSlots = 256;
constexpr int kTileRing = 16;                     // published work items a role may lag behind
__device__ int g_tc2_sched[kSchedSlots * 2];
constexpr int kTraceSteps = 256;
__device__ long long* g_tc2_trace = nullptr;
__device__ __forceinline__ void trace(long long* tr, int role, uint32_t step, int which) {
  if (tr != nullptr && step < kTraceSteps) {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    tr[((int64_t)role * kTraceSteps + step) * 2 + which] = t;
  }
}

#ifndef B200RL_TC2_WIDE_MAX_BN
#define B200RL_TC2_WIDE_MAX_BN 128
#endif
template <int BN, int PASSES, bool A_EXACT>
struct Layout {
  static constexpr int kATile = kBM * 128;
  static constexpr int kBTile = BN * 128;
  static constexpr int kNumA = (PASSES == 3 && !A_EXACT) ? 2 : 1;
  static constexpr int kNumB = PASSES == 3 ? 2 : 1;
  static constexpr int kRawA = A_EXACT ? kBM * kBK : 0;   // uint8 staging, expanded into plane A
  static constexpr int kStage = kNumA * kATile + kNumB * kBTile + kRawA;
  static constexpr int kBudget = 196 * 1024;
  static constexpr int kStages = (kBudget / kStage) > 8 ? 8 : (kBudget / kStage);
  // WIDE: the hi and lo planes of B sit side by side as ONE 2*BN-column operand, so that
  // A_hi x [B_hi | B_lo] is a single MMA of N = 2 BN into two accumulator column sets which the
  // epilogue adds.  The run-5 trace shows ~90 cycles per 128 x N x 8 TF32 MMA for N = 32, 64 and
  // 128 alike (the instruction is bound by its A-operand read / fixed latency, not by N), so a
  // 3xTF32 K step costs 2 MMAs instead of 3 and an exact-A step 1 instead of 2.
  static constexpr bool kWide = PASSES == 3 && BN <= B200RL_TC2_WIDE_MAX_BN;
  static constexpr int kAccCols = kWide ? 2 * BN : BN;     // TMEM columns of one accumulator
  static constexpr int kBarBytes = 512;
  static_assert(kStages + 4 <= kTileRing, "tile ring shorter than the deepest role lag");
  static constexpr int kBytes = kStages * kStage + 1024 /*alignment slack*/ + kBarBytes + BN * 4;
  static_assert(kStage % 1024 == 0, "stage planes must stay 1024 B aligned");
  static_assert(kStages >= 2, "at least two stages");
};

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes)
               : "memory");
}
__device__ __forceinline__ void cp_async_arrive(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(addr)
               : "memory");
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]),
        "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7])
      : "r"(taddr));
}
// one out-of-line body instead of 16 inlined tanhf expansions per epilogue step
__device__ __noinline__ float act_tanh(float x) { return tanhf(x); }
__device__ __forceinline__ float tf32_hi(float x) {
  return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
}

// Run-10 ncu source page of conv1.fwd: 2850 warp instructions per K block per CTA (70 % of the
// four schedulers' issue slots), of which a quarter were mbarrier polls (test_wait spins of the
// converters, nanosleep polls of the eight epilogue warps).  mbarrier.try_wait suspends the warp in
// hardware until the phase flips (or a time limit passes), so waiting roles stop taking issue slots
// from the loader / converter warps of their scheduler.  bit 6 of the flags: poll with test_wait
// as before (A/B switch).
__device__ __forceinline__ void mbar_wait_hw(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity, bool poll) {
  if (!poll) {
    mbar_wait_hw(bar, parity);
    return;
  }
  uint32_t done;
  int polls = 0;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (!done && ++polls > 4) __nanosleep(64);
  } while (!done);
}
__device__ __forceinline__ void mbar_wait_tight(uint32_t bar, uint32_t parity, bool poll) {
  if (poll) mbar_wait(bar, parity);
  else mbar_wait_hw(bar, parity);
}

struct Work {
  int64_t m0, n0, kb, ke;
  int split, nkb;
  bool first_m, second;
};
// Two problems of identical shape in one launch (DQN: the online network on obs[:, 0] and the
// target network on obs[:, T-1] -- same layers, different inputs and weights): m-tiles
// [tiles_m1, 2 tiles_m1) belong to the second problem, whose operands / outputs sit at fixed
// offsets from the first one's.  One launch instead of two saves the exposed fill + drain of a
// kernel boundary (~4-5 us on these layers) and halves the tile-count rounding loss.
struct PairArgs {
  int64_t tiles_m1;          // m-tiles of ONE problem (== tiles_m when the launch is not a pair)
  int64_t a_delta, b_delta;  // BYTES from the first problem's operand base to the second's
  int64_t c_delta, bias_delta;  // ELEMENTS between the outputs / biases
};
__device__ __forceinline__ Work decode_work(int64_t w, int64_t tiles_m, int64_t tiles_n, int BN,
                                            int64_t K, int64_t k_per_split, int64_t tiles_m1) {
  Work o;
  // 32-bit arithmetic (the host checks tiles * splits < 2^31): a 64-bit division is a call
  const uint32_t tiles_mn = (uint32_t)(tiles_m * tiles_n), wi = (uint32_t)w, tn_ = (uint32_t)tiles_n;
  const uint32_t split = wi / tiles_mn, rem = wi - split * tiles_mn;
  uint32_t tm = rem / tn_;
  const uint32_t tn = rem - tm * tn_;                           // n fastest: neighbours share A rows
  o.second = tm >= (uint32_t)tiles_m1;
  if (o.second) tm -= (uint32_t)tiles_m1;
  o.split = (int)split;
  o.m0 = (int64_t)tm * kBM;
  o.n0 = (int64_t)tn * BN;
  o.kb = (int64_t)split * k_per_split;
  o.ke = (o.kb + k_per_split < K) ? o.kb + k_per_split : K;
  o.nkb = (int)((o.ke - o.kb + kBK - 1) / kBK);
  o.first_m = tm == 0;
  return o;
}

// ---- loaders ------------------------------------------------------------------------------------
// K-contiguous fp32 view, ROWS x 32 tile: thread t owns chunk j = t & 7 (4 consecutive k) of rows
// (t >> 3) + 32 i.  sw128(r0 + 32 i, j) = sw128(r0, j) + 4096 i.  Row base POINTERS are hoisted per
// tile; a K block costs one k_off and, per chunk, one 64-bit add + the LDGSTS.
template <int ROWS, class V>
struct LoadKContigF32 {
  static constexpr int RPP = kLoaderThreads / 8;   // rows per pass
  static constexpr int NR = ROWS / RPP;
  const char* rowp[NR];                            // element (row, 0); rows past the edge: row 0
  uint32_t ok, dst0;
  int j;
  __device__ __forceinline__ void begin_tile(const V& v, int64_t row0, int64_t row_limit, int t,
                                             int64_t delta) {
    j = t & 7;
    const int r0 = t >> 3;
    dst0 = sw128((uint32_t)r0, (uint32_t)j);
    ok = 0;
#pragma unroll
    for (int i = 0; i < NR; ++i) {
      const int64_t r = row0 + r0 + RPP * i;
      const bool in = r < row_limit;
      rowp[i] = reinterpret_cast<const char*>(v.addr(in ? v.row_off(r) : 0)) + delta;
      ok |= (in ? 1u : 0u) << i;
    }
  }
  __device__ __forceinline__ void issue(const V& v, uint32_t plane, int64_t k0, int64_t ke) {
    const int64_t k = k0 + 4 * j;
    const bool kin = k < ke;                       // K % 4 == 0: a chunk is all in or all out
    const int64_t kbytes = kin ? v.k_off(k) * (int64_t)sizeof(float) : 0;
#pragma unroll
    for (int i = 0; i < NR; ++i)
      cp_async16(plane + dst0 + (RPP * 128u) * i, rowp[i] + kbytes, (kin && ((ok >> i) & 1u)) ? 16u : 0u);
  }
};

// MN-major fp32 view (the M/N index is contiguous in memory), 32 x ROWS tile: thread t owns row
// chunk cm = t % CPR (rows 4cm..4cm+3) at k-rows t / CPR + KSTEP i; the shared-memory offsets of
// its chunks are fixed for the whole kernel.  Linear views (k_off = k * ld) step their pointer;
// the conv filter-gradient view needs a full (n, oy, ox) decode per k: lane l computes it for
// k0 + l once and the offsets are fetched by shuffle.
template <int ROWS, class V, int LROWS = ROWS>
struct LoadMnF32 {                                 // LROWS: rows of the shared-memory tile layout
  static constexpr int CPR = ROWS / 4;
  static constexpr int KSTEP = kLoaderThreads / CPR;
  static constexpr int NC = 32 / KSTEP;            // chunks per thread
  const char* rowp;
  uint32_t dst[NC];
  bool ok;
  int kk0;
  __device__ __forceinline__ void begin_tile(const V& v, int64_t row0, int64_t row_limit, int t,
                                             int64_t delta) {
    const int cm = t % CPR;
    kk0 = t / CPR;
    const int64_t r = row0 + 4 * cm;
    ok = r < row_limit;                            // rows % 4 == 0 (host check)
    rowp = reinterpret_cast<const char*>(v.addr(ok ? v.row_off(r) : 0)) + delta;
#pragma unroll
    for (int i = 0; i < NC; ++i) dst[i] = mn128<LROWS>((uint32_t)cm, (uint32_t)(kk0 + KSTEP * i));
  }
  __device__ __forceinline__ void issue(const V& v, uint32_t plane, int64_t k0, int64_t ke) {
    if constexpr (V::kLinearK) {
      const int64_t step = v.k_stride() * (int64_t)sizeof(float);
      const char* p = rowp + (k0 + kk0) * step;
#pragma unroll
      for (int i = 0; i < NC; ++i) {
        const bool in = ok && (k0 + kk0 + KSTEP * i < ke);
        cp_async16(plane + dst[i], in ? p + (int64_t)(KSTEP * i) * step : rowp, in ? 16u : 0u);
      }
    } else {
      const int lane = threadIdx.x & 31;
      const int64_t my_koff = (k0 + lane < ke) ? v.k_off(k0 + lane) : 0;
#pragma unroll
      for (int i = 0; i < NC; ++i) {
        const int kk = kk0 + KSTEP * i;
        const int64_t koff = __shfl_sync(0xffffffffu, my_koff, kk);
        const bool in = ok && (k0 + kk < ke);
        cp_async16(plane + dst[i], rowp + (in ? koff : 0) * (int64_t)sizeof(float), in ? 16u : 0u);
      }
    }
  }
};

// K-contiguous uint8 im2col view (conv1 forward): raw tile [128 rows][32 B]; thread t copies
// 16-byte half t & 1 of row t >> 1 (one ky row of the patch = 32 contiguous bytes).  The halves of
// rows with bit 2 set are swapped (kept from the 128-thread converter; harmless).
template <class V>
struct LoadKContigU8 {
  int64_t roff;
  bool ok;
  uint32_t dst;
  int h;
  int64_t delta;
  __device__ __forceinline__ void begin_tile(const V& v, int64_t row0, int64_t row_limit, int t,
                                             int64_t delta_) {
    delta = delta_;
    const int row = t >> 1;
    h = t & 1;
    const int64_t r = row0 + row;
    ok = r < row_limit;
    roff = ok ? v.row_off(r) : 0;
    const uint32_t sw = (uint32_t)(row >> 2) & 1u;
    dst = (uint32_t)row * 32u + (((uint32_t)h ^ sw) << 4);
  }
  __device__ __forceinline__ void issue(const V& v, uint32_t raw, int64_t k0, int64_t ke) {
    const int64_t k = k0 + 16 * h;
    const bool in = ok && k < ke;                  // K % 16 == 0 (host check)
    cp_async16(raw + dst, reinterpret_cast<const char*>(v.addr(in ? roff + v.k_off(k) : 0)) + delta,
               in ? 16u : 0u);
  }
};

// MN-major uint8 view (conv1 filter gradient): raw tile [32 k][128 B]; the 128 patch indices of a
// k-row are 128/(KW*C) ky segments of contiguous bytes; thread t copies 16-byte chunk c = t & 7 of
// k-row t >> 3.
template <class V>
struct LoadMnU8 {
  int64_t roff;
  bool ok;
  int c, kk0;
  int64_t delta;
  __device__ __forceinline__ void begin_tile(const V& v, int64_t row0, int64_t row_limit, int t,
                                             int64_t delta_) {
    delta = delta_;
    c = t & 7;
    kk0 = t >> 3;
    const int64_t r = row0 + 16 * c;
    ok = r < row_limit;                            // rows % 16 == 0 (host check)
    roff = ok ? v.row_off(r) : 0;
  }
  __device__ __forceinline__ void issue(const V& v, uint32_t raw, int64_t k0, int64_t ke) {
    const int lane = threadIdx.x & 31;
    const int64_t my_koff = (k0 + lane < ke) ? v.k_off(k0 + lane) : 0;
    const int kk = kk0;
    const int64_t koff = __shfl_sync(0xffffffffu, my_koff, kk);
    const bool in = ok && (k0 + kk < ke);
    // slot c ^ 2(kk & 3): see convert_u8_mn
    cp_async16(raw + (uint32_t)kk * 128u + (((uint32_t)c ^ (((uint32_t)kk & 3u) << 1)) << 4),
               reinterpret_cast<const char*>(v.addr(in ? roff + koff : 0)) + delta, in ? 16u : 0u);
  }
};

// Plain row-major 2-D fp32 operand (ARow / BCol: dense inputs, dY, W^T): ONE thread issues ONE
// cp.async.bulk.tensor (TMA, SASS UTMALDG) per K block for the whole ROWS x 32 tile; the tensor
// map's SWIZZLE_128B mode writes exactly the K-major layout the MMA descriptors expect, rows / k
// past the matrix edge are zero-filled by the unit, and completion is counted in bytes on the same
// mbarrier the other loader threads arrive on.
template <int ROWS>
struct LoadTma2D {
  int32_t row0;
  __device__ __forceinline__ void begin_tile(int64_t r0) { row0 = (int32_t)r0; }
  __device__ __forceinline__ void issue(const CUtensorMap* tm, uint32_t plane, int64_t k0, uint32_t bar) {
    if ((threadIdx.x & (kLoaderThreads - 1)) == 0) {
      asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar),
                   "r"((uint32_t)(ROWS * kBK * sizeof(float)))
                   : "memory");
      asm volatile(
          "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
          "[%0], [%1, {%2, %3}], [%4];" ::"r"(plane),
          "l"(reinterpret_cast<uint64_t>(tm)), "r"((int32_t)k0), "r"(row0), "r"(bar)
          : "memory");
    }
  }
};

template <int ROWS, class V, bool KCONTIG = V::kKContig, bool EXACT = V::kExact>
struct LoaderFor;
template <int ROWS, class V>
struct LoaderFor<ROWS, V, true, false> { using type = LoadKContigF32<ROWS, V>; };
template <int ROWS, class V>
struct LoaderFor<ROWS, V, false, false> { using type = LoadMnF32<ROWS, V>; };
template <int ROWS, class V>
struct LoaderFor<ROWS, V, true, true> { using type = LoadKContigU8<V>; };
template <int ROWS, class V>
struct LoaderFor<ROWS, V, false, true> { using type = LoadMnU8<V>; };

// ---- converters ---------------------------------------------------------------------------------
// fp32 plane of `bytes` bytes: hi in place, lo at +lo_off; 128 threads, 16 B per thread per step.
template <bool WITH_LO>
__device__ __forceinline__ void convert_f32(uint32_t plane, uint32_t lo_off, int bytes, int t,
                                            bool raw_hi, float4& colsum, bool do_colsum) {
#pragma unroll 4
  for (int off = t * 16; off < bytes; off += kConvThreads * 16) {
    const float4 v = lds128(plane + off);
    float4 h;
    h.x = tf32_hi(v.x); h.y = tf32_hi(v.y); h.z = tf32_hi(v.z); h.w = tf32_hi(v.w);
    if (!raw_hi) sts128(plane + off, h);
    if (WITH_LO) sts128(plane + lo_off + off, make_float4(v.x - h.x, v.y - h.y, v.z - h.z, v.w - h.w));
    if (do_colsum) { colsum.x += v.x; colsum.y += v.y; colsum.z += v.z; colsum.w += v.w; }
  }
}
// MN-major B tile of the WIDE layout: per 4-row k atom, the BN/32 hi atoms are followed by the
// BN/32 lo atoms (mn128<2 BN> with the lo rows at cm + BN/4), i.e. lo = hi + BN * 16 bytes.
template <int BN>
__device__ __forceinline__ void convert_f32_mn_wide(uint32_t plane, int t, bool raw_hi,
                                                    float4& colsum, bool do_colsum) {
#pragma unroll 4
  for (int i = t; i < BN * 8; i += kConvThreads) {
    const uint32_t off = (uint32_t)(i / BN) * (2u * BN * 16u) + (uint32_t)(i % BN) * 16u;
    const float4 v = lds128(plane + off);
    float4 h;
    h.x = tf32_hi(v.x); h.y = tf32_hi(v.y); h.z = tf32_hi(v.z); h.w = tf32_hi(v.w);
    if (!raw_hi) sts128(plane + off, h);
    sts128(plane + off + BN * 16u, make_float4(v.x - h.x, v.y - h.y, v.z - h.z, v.w - h.w));
    if (do_colsum) { colsum.x += v.x; colsum.y += v.y; colsum.z += v.z; colsum.w += v.w; }
  }
}
// 4 packed uint8 -> 4 floats, exactly: PRMT builds 0x4B0000bb = 2^23 + b, one FADD removes the
// 2^23 (2 full-rate instructions per pixel instead of shift + mask + I2F)
__device__ __forceinline__ void u8x4_to_f32(uint32_t w, float4& o) {
  o.x = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540)) - 8388608.f;
  o.y = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7541)) - 8388608.f;
  o.z = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7542)) - 8388608.f;
  o.w = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7543)) - 8388608.f;
}
// raw [128 rows][32 B] uint8 -> K-major SWIZZLE_128B fp32 tile: thread t expands 16-byte half
// t & 1 of row t >> 1 (a quarter-warp stores 4 rows x chunks {q, q + 4}: eight distinct slots)
__device__ __forceinline__ void convert_u8_kcontig(uint32_t raw, uint32_t plane, int t) {
  const uint32_t row = (uint32_t)t >> 1, h = (uint32_t)t & 1u;
  const uint32_t sw = (row >> 2) & 1u;
  uint4 p;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(p.x), "=r"(p.y), "=r"(p.z), "=r"(p.w)
               : "r"(raw + row * 32u + ((h ^ sw) << 4))
               : "memory");
  const uint32_t w[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float4 o;
    u8x4_to_f32(w[q], o);
    sts128(plane + sw128(row, 4u * h + (uint32_t)q), o);
  }
}
// raw [32 k][128 B] uint8 -> MN-major fp32 tile (128 rows).  Chunk (kk, c) = the 16 patch
// elements 16c..16c+15 at reduction index kk sits in 16-byte slot c ^ 2(kk & 3) of raw row kk
// (LoadMnU8 writes it there).  A quarter-warp = 4 consecutive kk x 2 neighbouring chunks: its
// eight 16-byte reads hit eight different slots, and because lanes with odd c walk their four
// float4 sub-chunks in the order q ^ 1, its eight stores land in the eight different 16-byte
// slots of one 512 B atom of the SWIZZLE_128B_BASE32B layout -- no bank conflicts on either side.
__device__ __forceinline__ void convert_u8_mn(uint32_t raw, uint32_t plane, int t) {
  const uint32_t kin = (uint32_t)t & 3u, cb = ((uint32_t)t >> 2) & 1u;
  const uint32_t c = ((((uint32_t)t >> 3) & 3u) << 1) | cb, kq = ((uint32_t)t >> 5) & 7u;
  {
    const uint32_t kk = (kq << 2) | kin;
    uint4 p;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(p.x), "=r"(p.y), "=r"(p.z), "=r"(p.w)
                 : "r"(raw + kk * 128u + ((c ^ (kin << 1)) << 4))
                 : "memory");
    // sub-chunk order q ^ cb without dynamic register indexing
    const uint32_t w0 = cb ? p.y : p.x, w1 = cb ? p.x : p.y, w2 = cb ? p.w : p.z, w3 = cb ? p.z : p.w;
    const uint32_t w[4] = {w0, w1, w2, w3};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float4 o;
      u8x4_to_f32(w[q], o);
      sts128(plane + mn128<kBM>(4u * c + ((uint32_t)q ^ cb), kk), o);
    }
  }
}

// ---- the kernel ---------------------------------------------------------------------------------
template <int BN, int PASSES, int EPI, class AL, class BL>
__global__ void __launch_bounds__(kThreads, 1)
    tc2_gemm_kernel(const AL a, const BL b, const EpiArgs epi, float* __restrict__ C,
                    const float* __restrict__ bias, int64_t M, int64_t N, int64_t K, int act,
                    int beta, int splits, int64_t k_per_split, float* __restrict__ ws,
                    float out_scale, int64_t tiles_m, int64_t tiles_n, int epi_warps,
                    int sched_slot, const PairArgs pair,
                    const __grid_constant__ CUtensorMap tmA,
                    const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmA2,
                    const __grid_constant__ CUtensorMap tmB2) {
  using L = Layout<BN, PASSES, AL::kExact>;
  constexpr int S = L::kStages;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t smem_base = smem_addr(smem);
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + S * L::kStage);
  unsigned long long* raw_full = bars;            // loaders' cp.async landed
  unsigned long long* conv_full = bars + S;       // converters done -> MMA may read
  unsigned long long* empty = bars + 2 * S;       // MMAs of the stage retired -> loaders
  unsigned long long* acc_full = bars + 3 * S;    // [2] accumulator complete -> epilogue
  unsigned long long* acc_empty = acc_full + 2;   // [2] epilogue drained it -> MMA
  unsigned long long* tile_full = acc_empty + 2;  // [kTileRing] work item published
  int* tile_slot = reinterpret_cast<int*>(tile_full + kTileRing);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tile_slot + kTileRing);
  float* scol = reinterpret_cast<float*>(smem + S * L::kStage + L::kBarBytes);   // [BN] column sums
  static_assert((3 * 8 + 4 + kTileRing) * 8 + kTileRing * 4 + 8 <= L::kBarBytes, "barrier block too small");

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  pdl_launch_dependents();
  if (tid == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(smem_addr(&raw_full[s]), kLoaderThreads);
      mbar_init(smem_addr(&conv_full[s]), kConvThreads / 32);
      mbar_init(smem_addr(&empty[s]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_addr(&acc_full[i]), 1);
      mbar_init(smem_addr(&acc_empty[i]), (uint32_t)epi_warps);
    }
    for (int i = 0; i < kTileRing; ++i) mbar_init(smem_addr(&tile_full[i]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < BN) scol[tid] = 0.f;
  constexpr bool kWide = L::kWide;
  constexpr int kCols = 2 * L::kAccCols;           // two accumulators; power of two >= 64
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_addr(tmem_slot)),
                 "n"(kCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                                      // nothing above touched global memory

  const int64_t total = tiles_m * tiles_n * (int64_t)splits;
  long long* const tr = blockIdx.x == 0 ? g_tc2_trace : nullptr;
  const bool poll = (g_tc2_flags & 64) != 0;
  // Work items: the first one of a CTA is blockIdx.x; with a scheduler slot the following ones come
  // from a global counter (loader thread 0 fetches one item ahead and publishes each item in a
  // shared-memory ring that every role reads), so a CTA that starts late -- its SM was busy with a
  // collective or a kernel of the other stream -- simply takes fewer tiles instead of holding the
  // whole launch back by its statically assigned share.
  int* const sched = sched_slot >= 0 ? g_tc2_sched + 2 * sched_slot : nullptr;
  auto next_tile = [&](uint32_t tq) -> int64_t {
    if (sched == nullptr) {
      const int64_t w = (int64_t)blockIdx.x + (int64_t)tq * gridDim.x;
      return w < total ? w : -1;
    }
    const uint32_t slot = tq & (kTileRing - 1);
    mbar_wait_hw(smem_addr(&tile_full[slot]), (tq / kTileRing) & 1u);
    return *reinterpret_cast<volatile int*>(&tile_slot[slot]);
  };
  constexpr bool kLoA = PASSES == 3 && !AL::kExact;
  constexpr bool kLoB = PASSES == 3;
  constexpr uint32_t kOffB = L::kNumA * L::kATile;
  constexpr uint32_t kOffRaw = kOffB + L::kNumB * L::kBTile;

  if (warp < kLoaderThreads / 32) {
    // ======================= loaders =======================
    typename LoaderFor<kBM, AL>::type la;
    typename std::conditional<kWide && !BL::kKContig, LoadMnF32<BN, BL, 2 * BN>,
                              typename LoaderFor<BN, BL>::type>::type lb;
    LoadTma2D<kBM> ta;                             // used instead of la / lb for plain 2-D operands
    LoadTma2D<BN> tb;
    const bool use_tma = (g_tc2_flags & 4) == 0;   // bit 2: cp.async loaders for those as well (A/B)
    const bool no_load = (g_tc2_flags & 8) != 0;
    uint32_t it = 0, ring_s = 0, ring_ph = 0;      // stage / phase of K block `it` without a division
    int64_t fetched = blockIdx.x;                   // scheduler (thread 0): the item to publish next
    for (uint32_t tq = 0;; ++tq) {
      if (sched != nullptr && tid == 0) {
        const int v = fetched < total ? (int)fetched : -1;
        const uint32_t slot = tq & (kTileRing - 1);
        *reinterpret_cast<volatile int*>(&tile_slot[slot]) = v;
        mbar_arrive(smem_addr(&tile_full[slot]));
        if (v >= 0) {
          fetched = (int64_t)gridDim.x + atomicAdd(sched, 1);   // used one tile later
        } else if (atomicAdd(sched + 1, 1) == (int)gridDim.x - 1) {
          atomicExch(sched, 0);                     // every CTA has drawn its last item: leave the
          atomicExch(sched + 1, 0);                 // slot zeroed for its next launch
        }
      }
      const int64_t w = next_tile(tq);
      if (w < 0) break;
      const Work wk = decode_work(w, tiles_m, tiles_n, BN, K, k_per_split, pair.tiles_m1);
      if (AL::kTma2D && use_tma) ta.begin_tile(wk.m0);
      else la.begin_tile(a, wk.m0, M, tid, wk.second ? pair.a_delta : 0);
      if (BL::kTma2D && use_tma) tb.begin_tile(wk.n0);
      else lb.begin_tile(b, wk.n0, N, tid, wk.second ? pair.b_delta : 0);
#pragma unroll 1
      for (int kbi = 0; kbi < wk.nkb; ++kbi, ++it) {
        const uint32_t s = ring_s, ph = ring_ph;
        if (++ring_s == S) { ring_s = 0; ring_ph ^= 1u; }
        mbar_wait_relaxed(smem_addr(&empty[s]), ph ^ 1u, poll);
        if (tid == 0) trace(tr, 0, it, 0);
        const uint32_t st = smem_base + s * L::kStage;
        const int64_t k0 = wk.kb + (int64_t)kbi * kBK;
        const uint32_t bar = smem_addr(&raw_full[s]);
        if (!no_load) {
          if (AL::kTma2D && use_tma) ta.issue(wk.second ? &tmA2 : &tmA, st, k0, bar);
          else la.issue(a, AL::kExact ? st + kOffRaw : st, k0, wk.ke);
          if (BL::kTma2D && use_tma) tb.issue(wk.second ? &tmB2 : &tmB, st + kOffB, k0, bar);
          else lb.issue(b, st + kOffB, k0, wk.ke);
        }
        cp_async_arrive(smem_addr(&raw_full[s]));
        if (tid == 0) trace(tr, 0, it, 1);
      }
    }
  } else if (warp < kMmaWarp) {
    // ======================= converters =======================
    const int t = tid - kLoaderThreads;
    const bool raw_hi = (g_tc2_flags & 1) == 0;
    const bool no_conv = (g_tc2_flags & 16) != 0;
    uint32_t it = 0, ring_s = 0, ring_ph = 0;
    for (uint32_t tq = 0;; ++tq) {
      const int64_t w = next_tile(tq);
      if (w < 0) break;
      const Work wk = decode_work(w, tiles_m, tiles_n, BN, K, k_per_split, pair.tiles_m1);
      const bool do_colsum = EPI == EPI_ATOMIC && !BL::kKContig && epi.colsum != nullptr && wk.first_m;
      float4 csum = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
      for (int kbi = 0; kbi < wk.nkb; ++kbi, ++it) {
        const uint32_t s = ring_s, ph = ring_ph;
        if (++ring_s == S) { ring_s = 0; ring_ph ^= 1u; }
        mbar_wait_tight(smem_addr(&raw_full[s]), ph, poll);
        if (t == 0) trace(tr, 1, it, 0);
        const uint32_t st = smem_base + s * L::kStage;
        float4 none = make_float4(0.f, 0.f, 0.f, 0.f);
        if (no_conv) {
        } else if (AL::kExact) {
          if (AL::kKContig) convert_u8_kcontig(st + kOffRaw, st, t);
          else convert_u8_mn(st + kOffRaw, st, t);
        } else if (PASSES == 3 || !raw_hi) {
          convert_f32<kLoA>(st, L::kATile, L::kATile, t, raw_hi, none, false);
        }
        if (no_conv) {
        } else if (kWide && !BL::kKContig)
          convert_f32_mn_wide<BN>(st + kOffB, t, raw_hi, csum, do_colsum);
        else if (PASSES == 3 || !raw_hi || do_colsum)
          convert_f32<kLoB>(st + kOffB, L::kBTile, L::kBTile, t, raw_hi, csum, do_colsum);
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_addr(&conv_full[s]));
        if (t == 0) trace(tr, 1, it, 1);
      }
      if (do_colsum) {
        // Every chunk of a thread covers the same 4 columns (the MN-major atom layout repeats
        // with the thread stride): decode them from the thread's first byte offset.
        const uint32_t off = (uint32_t)t * 16u, within = off & 511u;
        const uint32_t kin = within >> 7, blk = (within & 127u) >> 4;
        const uint32_t c = (((blk >> 1) ^ kin) << 1) | (blk & 1u);
        const uint32_t cm = ((off >> 9) % (BN / 32)) * 8u + c;
        atomicAdd(&scol[4 * cm + 0], csum.x);
        atomicAdd(&scol[4 * cm + 1], csum.y);
        atomicAdd(&scol[4 * cm + 2], csum.z);
        atomicAdd(&scol[4 * cm + 3], csum.w);
        asm volatile("bar.sync 2, %0;" ::"n"(kConvThreads) : "memory");
        if (t < BN) {
          const float v = scol[t];
          scol[t] = 0.f;
          if (wk.n0 + t < N) atomicAdd(epi.colsum + wk.n0 + t, v);
        }
        asm volatile("bar.sync 2, %0;" ::"n"(kConvThreads) : "memory");
      }
    }
  } else if (warp == kMmaWarp) {
    // ======================= MMA issuer =======================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(BN, !AL::kKContig, !BL::kKContig);
      constexpr uint32_t idesc_w = make_idesc(2 * BN, !AL::kKContig, !BL::kKContig);
      constexpr int kBRows = kWide ? 2 * BN : BN;   // rows of the MN-major B tile layout
      // One thread issues every MMA, so its scalar instruction stream IS the K-loop rate once the
      // operands arrive (run 4 trace: 560 ns per K block, ~30 instructions per MMA, most of them
      // rebuilding shared-memory descriptors).  Everything but the 14-bit start-address field of a
      // descriptor is constant: keep the constants, and advance the start fields (16-byte units)
      // with 32-bit adds.
      constexpr uint32_t kaStep = AL::kKContig ? 2u : (2u * (kBM / 32) * 512u) >> 4;   // per K = 8
      constexpr uint32_t kbStep = BL::kKContig ? 2u : (2u * (kBRows / 32) * 512u) >> 4;
      constexpr uint32_t kStageStep = (uint32_t)L::kStage >> 4;
      const uint64_t dA = AL::kKContig ? make_desc(0) : make_desc_mn(0, (kBM / 32) * 512u);
      const uint64_t dB = BL::kKContig ? make_desc(0) : make_desc_mn(0, (kBRows / 32) * 512u);
      const uint32_t fa_hi = smem_base >> 4, fa_lo = (smem_base + L::kATile) >> 4;
      const uint32_t fb_hi = (smem_base + kOffB) >> 4, fb_lo = (smem_base + kOffB + L::kBTile) >> 4;
      const bool no_mma = (g_tc2_flags & 32) != 0;
      uint32_t it = 0, tl = 0, ring_s = 0, ring_ph = 0;
      for (;; ++tl) {
        const int64_t w = next_tile(tl);
        if (w < 0) break;
        const Work wk = decode_work(w, tiles_m, tiles_n, BN, K, k_per_split, pair.tiles_m1);
        const uint32_t buf = tl & 1u;
        mbar_wait_tight(smem_addr(&acc_empty[buf]), ((tl >> 1) & 1u) ^ 1u, poll);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t tmem_d = tmem_base + buf * L::kAccCols;
#pragma unroll 1
        for (int kbi = 0; kbi < wk.nkb; ++kbi, ++it) {
          const uint32_t s = ring_s, ph = ring_ph;
        if (++ring_s == S) { ring_s = 0; ring_ph ^= 1u; }
          mbar_wait_tight(smem_addr(&conv_full[s]), ph, poll);
          trace(tr, 2, it, 0);
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic stores -> async proxy
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t so = s * kStageStep;
          const uint32_t first = kbi == 0 ? 0u : 1u;
#pragma unroll
          for (int ks = 0; ks < kBK / 8; ++ks) {
            if (no_mma) break;
            const uint32_t oa = so + (uint32_t)ks * kaStep, ob = so + (uint32_t)ks * kbStep;
            const uint32_t acc0 = ks == 0 ? first : 1u;
            if (kWide && AL::kExact) {
              tc_mma_tf32(tmem_d, dA + (fa_hi + oa), dB + (fb_hi + ob), idesc_w, acc0);
            } else if (kWide) {
              // columns [0, BN): A_hi B_hi + A_lo B_hi; columns [BN, 2 BN): A_hi B_lo
              tc_mma_tf32(tmem_d, dA + (fa_hi + oa), dB + (fb_hi + ob), idesc_w, acc0);
              tc_mma_tf32(tmem_d, dA + (fa_lo + oa), dB + (fb_hi + ob), idesc, 1u);
            } else if (PASSES == 3 && AL::kExact) {
              tc_mma_tf32(tmem_d, dA + (fa_hi + oa), dB + (fb_lo + ob), idesc, acc0);
              tc_mma_tf32(tmem_d, dA + (fa_hi + oa), dB + (fb_hi + ob), idesc, 1u);
            } else if (PASSES == 3) {
              tc_mma_tf32(tmem_d, dA + (fa_lo + oa), dB + (fb_hi + ob), idesc, acc0);
              tc_mma_tf32(tmem_d, dA + (fa_hi + oa), dB + (fb_lo + ob), idesc, 1u);
              tc_mma_tf32(tmem_d, dA + (fa_hi + oa), dB + (fb_hi + ob), idesc, 1u);
            } else {
              tc_mma_tf32(tmem_d, dA + (fa_hi + oa), dB + (fb_hi + ob), idesc, acc0);
            }
          }
          tc_commit(smem_addr(&empty[s]));
          trace(tr, 2, it, 1);
        }
        tc_commit(smem_addr(&acc_full[buf]));
      }
    }
    __syncwarp();
  } else if (warp < kFirstEpiWarp + epi_warps) {
    // ======================= epilogue =======================
    const int q = warp & 3;                        // TMEM lane quadrant this warp may read
    const int chalf = (warp - kFirstEpiWarp) >> 2; // which part of the tile's columns it drains
    const int kColsPerWarp = BN / (epi_warps >> 2);
    uint32_t tl = 0;
    for (;; ++tl) {
      const int64_t w = next_tile(tl);
      if (w < 0) break;
      const Work wk = decode_work(w, tiles_m, tiles_n, BN, K, k_per_split, pair.tiles_m1);
      const uint32_t buf = tl & 1u;
      if (EPI == EPI_STORE && epi.mask.y != nullptr && splits == 1) {
        // act' mask rows of this tile: start them towards L2 while the accumulator is still being
        // produced (run 13: the mask loads sat behind every tcgen05.ld on the PPO dX GEMM)
        const int64_t mm = wk.m0 + (warp & 3) * 32 + lane;
        if (mm < M) {
          const float* yrow = epi.mask.y + mm * epi.mask.ld + wk.n0;
          const int c0 = ((warp - kFirstEpiWarp) >> 2) * (BN / (epi_warps >> 2));
          for (int c = c0; c < c0 + BN / (epi_warps >> 2); c += 32)
            if (wk.n0 + c < N) asm volatile("prefetch.global.L2 [%0];" ::"l"(yrow + c));
        }
      }
      mbar_wait_relaxed(smem_addr(&acc_full[buf]), (tl >> 1) & 1u, poll);
      if (warp == kFirstEpiWarp && lane == 0) trace(tr, 3, tl, 0);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const int64_t m = wk.m0 + q * 32 + lane;
      float* const Cx = C + (wk.second ? pair.c_delta : 0);
      const float* const biasx = bias ? bias + (wk.second ? pair.bias_delta : 0) : nullptr;
      float* out = (splits > 1 && EPI == EPI_STORE)
                       ? ws + ((int64_t)(wk.second ? splits : 0) + wk.split) * M * N : Cx;
      const bool vec_out = (N & 3) == 0 && ((uintptr_t)out & 15) == 0;
      const bool final_pass = splits == 1;
      const bool vec_mask = (N & 3) == 0 && (epi.mask.ld & 3) == 0 && ((uintptr_t)epi.mask.y & 15) == 0;
      // col2im destination of this row (EPI_COL2IM): pos -> (n, oy, ox)
      float* cbase = nullptr;
      const float* ybase = nullptr;
      int64_t wc = 0;
      uint32_t ox = 0;
      if ((EPI == EPI_COL2IM || EPI == EPI_COL2IM_MERGE) && m < M) {
        uint32_t img, rem, oy;
        epi.g.d_ohow.divmod((uint32_t)m, img, rem);
        epi.g.d_ow.divmod(rem, oy, ox);
        wc = (int64_t)epi.g.W * epi.g.C;
        const int64_t in_off = (int64_t)oy * epi.g.stride * wc + (int64_t)ox * epi.g.stride * epi.g.C;
        cbase = epi.dx + (int64_t)img * epi.g.H * wc + in_off;
        if (epi.mask.y) ybase = epi.mask.y + (int64_t)img * epi.mask.ld + in_off;
      }
      if constexpr (EPI == EPI_COL2IM_MERGE) {
        // Neighbour pre-sum.  Output positions (oy, ox) and (oy, ox + 1) are consecutive rows m,
        // i.e. consecutive TMEM lanes, and patch column (ky, kx, ch) of the first addresses the same
        // input element as column (ky, kx - stride, ch) of the second: merge_cols = stride * C = 64
        // columns to the left, the other half of this 128-column tile.  Each warp therefore drains
        // a 16-column chunk of the low half together with its partner chunk of the high half, adds
        // its right neighbour's low values to its own high values with one shuffle per column, and
        // issues the low-half red only where no left neighbour took it (lane 0 of the warp, first
        // column of an image row): ~1.14 instead of 2 red.global.add.v4 per pair of 4-channel
        // groups for a 9-wide output.  act'(y) depends on the target only, so it is applied to
        // the merged sum.  The summation order of dX was never fixed (atomics).
        const bool row_ok = m < M;
        const bool take = row_ok && lane < 31 && m + 1 < M && ox + 1 < (uint32_t)epi.g.OW;
        const bool given = row_ok && lane > 0 && ox > 0;
        const uint32_t kwc = (uint32_t)(epi.g.KW * epi.g.C), wc32 = (uint32_t)wc;
        const int kLowPerWarp = 64 / (epi_warps >> 2);
        // accumulator columns [c, c + 8) of this lane's row (the two column sets of the WIDE layout
        // added); 8 instead of 16 columns per tcgen05.ld keeps the live set of the merged pass
        // within the register cap of an 800-thread CTA
        auto load8 = [&](int c, uint32_t (&r)[8]) {
          const uint32_t taddr =
              tmem_base + ((uint32_t)(q * 32) << 16) + buf * L::kAccCols + (uint32_t)c;
          tmem_ld8(taddr, r);
          if (kWide) {
            uint32_t r2[8];
            tmem_ld8(taddr + BN, r2);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int j = 0; j < 8; ++j)
              r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(r2[j]));
          } else {
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          }
        };
        auto red4 = [&](uint32_t off, float4 v) {
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(cbase + off),
                       "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                       : "memory");
        };
        auto masked = [&](float4 y, float4 v) {
          v.x = dact(y.x, v.x, epi.mask.act); v.y = dact(y.y, v.y, epi.mask.act);
          v.z = dact(y.z, v.z, epi.mask.act); v.w = dact(y.w, v.w, epi.mask.act);
          return v;
        };
#pragma unroll 1
        for (int c = chalf * kLowPerWarp; c < (chalf + 1) * kLowPerWarp; c += 16) {
          const uint32_t nb_lo = (uint32_t)wk.n0 + (uint32_t)c, nb_hi = nb_lo + 64u;
          if (nb_lo >= (uint32_t)N) break;         // N % 16 == 0: a chunk is all in or all out
          const bool hi_ok = nb_hi < (uint32_t)N;  // uniform over the warp
          uint32_t ky_lo, rr_lo;
          epi.g.d_kwc.divmod(nb_lo, ky_lo, rr_lo);
          const bool merge = hi_ok && rr_lo + 64u < kwc;   // partner chunk in the same ky row
          const bool need_lo = row_ok && !(merge && given);
          const bool need_hi = row_ok && hi_ok;
#pragma unroll
          for (int h = 0; h < 2; ++h) {            // 8 columns (two 4-channel groups) at a time
            // patch column -> (ky, kx * C + ch) -> offset into dX / the act' mask; the mask loads of
            // both chunks are issued BEFORE the accumulator reads so that their latency overlaps the
            // tcgen05.ld round trips and the shuffles (run 22: with one dependent load per group the
            // saved atomics were paid back in load latency)
            uint32_t off_lo[2], off_hi[2];
            float4 y_lo[2], y_hi[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              uint32_t ky, rr;
              epi.g.d_kwc.divmod(nb_lo + (uint32_t)(8 * h + 4 * j), ky, rr);
              off_lo[j] = ky * wc32 + rr;
              epi.g.d_kwc.divmod(nb_hi + (uint32_t)(8 * h + 4 * j), ky, rr);
              off_hi[j] = ky * wc32 + rr;
              if (ybase && need_lo) y_lo[j] = *reinterpret_cast<const float4*>(ybase + off_lo[j]);
              if (ybase && need_hi) y_hi[j] = *reinterpret_cast<const float4*>(ybase + off_hi[j]);
            }
            uint32_t lo[8];
            load8(c + 8 * h, lo);
            float t[8];                            // the right neighbour's low values
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float nbr = __shfl_down_sync(0xffffffffu, __uint_as_float(lo[j]), 1);
              t[j] = (merge && take) ? nbr : 0.f;
            }
            if (need_lo) {                         // (before the partner read: lo / y_lo die here)
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                float4 v = make_float4(__uint_as_float(lo[4 * j]), __uint_as_float(lo[4 * j + 1]),
                                       __uint_as_float(lo[4 * j + 2]), __uint_as_float(lo[4 * j + 3]));
                if (ybase) v = masked(y_lo[j], v);
                red4(off_lo[j], v);
              }
            }
            uint32_t hi[8];
            if (hi_ok) load8(c + 64 + 8 * h, hi);
            if (need_hi) {
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                float4 v = make_float4(__uint_as_float(hi[4 * j]) + t[4 * j],
                                       __uint_as_float(hi[4 * j + 1]) + t[4 * j + 1],
                                       __uint_as_float(hi[4 * j + 2]) + t[4 * j + 2],
                                       __uint_as_float(hi[4 * j + 3]) + t[4 * j + 3]);
                if (ybase) v = masked(y_hi[j], v);
                red4(off_hi[j], v);
              }
            }
          }
        }
      } else {
#pragma unroll 1
      for (int c = chalf * kColsPerWarp; c < (chalf + 1) * kColsPerWarp; c += 16) {
        uint32_t r[16];
        const uint32_t taddr =
            tmem_base + ((uint32_t)(q * 32) << 16) + buf * L::kAccCols + (uint32_t)c;
        tmem_ld16(taddr, r);
        if (kWide) {
          uint32_t r2[16];
          tmem_ld16(taddr + BN, r2);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
          for (int j = 0; j < 16; ++j)
            r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(r2[j]));
        } else {
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        }
        const int64_t nb = wk.n0 + c;
        if (m >= M || nb >= N) continue;
        if (EPI == EPI_COL2IM) {
          float4 y4[4];
          uint32_t off4[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {            // 4-channel groups: patch index -> (ky, kx*C + c)
            uint32_t ky, rr;
            epi.g.d_kwc.divmod((uint32_t)(nb + 4 * j), ky, rr);
            off4[j] = (uint32_t)(ky * wc + rr);
            if (ybase && nb + 4 * j < N) y4[j] = *reinterpret_cast<const float4*>(ybase + off4[j]);
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (nb + 4 * j >= N) break;
            float4 v = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
                                   __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
            if (ybase) {
              v.x = dact(y4[j].x, v.x, epi.mask.act); v.y = dact(y4[j].y, v.y, epi.mask.act);
              v.z = dact(y4[j].z, v.z, epi.mask.act); v.w = dact(y4[j].w, v.w, epi.mask.act);
            }
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(cbase + off4[j]),
                         "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                         : "memory");
          }
        } else if (EPI == EPI_ATOMIC) {
          float* dst = Cx + m * N + nb;
          if ((N & 3) == 0) {
#pragma unroll
            for (int j = 0; j < 16; j += 4) {
              if (nb + j >= N) break;
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + j),
                           "f"(__uint_as_float(r[j]) * out_scale),
                           "f"(__uint_as_float(r[j + 1]) * out_scale),
                           "f"(__uint_as_float(r[j + 2]) * out_scale),
                           "f"(__uint_as_float(r[j + 3]) * out_scale)
                           : "memory");
            }
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (nb + j < N) atomicAdd(dst + j, __uint_as_float(r[j]) * out_scale);
          }
        } else {
          float v[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]) * out_scale;
          if (final_pass) {
            const bool full = nb + 15 < N;
            if (biasx) {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] += (full || nb + j < N) ? __ldg(biasx + nb + j) : 0.f;
            }
            if (act == B200RL_ACT_RELU) {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
            } else if (act == B200RL_ACT_TANH) {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = act_tanh(v[j]);
            }
            if (epi.mask.y) {
              const float* yp = epi.mask.y + m * epi.mask.ld + nb;
              if (vec_mask) {                      // 4 x LDG.128 instead of 16 scalar loads per lane
#pragma unroll
                for (int j = 0; j < 16; j += 4) {
                  if (nb + j < N) {
                    const float4 y = *reinterpret_cast<const float4*>(yp + j);
                    v[j] = dact(y.x, v[j], epi.mask.act);
                    v[j + 1] = dact(y.y, v[j + 1], epi.mask.act);
                    v[j + 2] = dact(y.z, v[j + 2], epi.mask.act);
                    v[j + 3] = dact(y.w, v[j + 3], epi.mask.act);
                  }
                }
              } else {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                  if (full || nb + j < N) v[j] = dact(yp[j], v[j], epi.mask.act);
              }
            }
            if (beta) {
#pragma unroll
              for (int j = 0; j < 16; ++j)
                if (full || nb + j < N) v[j] += out[m * N + nb + j];
            }
          }
          float* dst = out + m * N + nb;
          if (vec_out) {
#pragma unroll
            for (int j = 0; j < 16; j += 4)
              if (nb + j < N)
                *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (nb + j < N) dst[j] = v[j];
          }
        }
      }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_addr(&acc_empty[buf]));
      if (warp == kFirstEpiWarp && lane == 0) trace(tr, 3, tl, 1);
    }
  }
  __syncthreads();
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "n"(kCols));
  }
}

}  // namespace tc2
}  // namespace b200rl
