// CDS_OP_CONV, tensor-core path (CDS_MATH_BF16_TC / CDS_MATH_TF32_TC): implicit-GEMM 1-D convolution on tcgen05 with the
// UNet block post-processing fused into the TMEM epilogue.  Template parameter TF32 selects the operand type: bf16
// activations / weights (kind::f16) or fp32 activations / weights read as TF32 (kind::tf32).  Everything about the operand
// tiles is expressed in BYTES: "KC" is the row width of a chunk in bf16-equivalents (row bytes / 2: 64 -> 128-byte rows,
// SWIZZLE_128B; 32 -> 64-byte rows, SWIZZLE_64B), i.e. KC channels of bf16 or KC/2 channels of fp32, and one MMA
// instruction always consumes 32 bytes of K (16 bf16 / 8 tf32).
//
//   D[128 rows x N] (fp32, TMEM) = sum over (tap, 64- or 32-channel chunk) of  A_tap[128 x KC] * W_tap[N x KC]^T
//
// * rows = 128/L whole trajectories x L positions.  The im2col never exists: the A tile of tap j is ONE TMA box
//   {KC channels, L positions, T trajectories} of the channels-last bf16 activation whose position coordinate starts at
//   j - pad; positions outside [0, L) are zero-filled by the TMA unit (out-of-bound fill), which is exactly the conv's
//   zero padding, and trajectories never bleed into each other because they are a separate tensor dimension.
// * W_tap is a TMA box {KC, N} of the bf16 weight packed [tap][C_out][C_in]; both operands land in shared memory in the
//   K-major SWIZZLE_128B (KC=64) / SWIZZLE_64B (KC=32) layout that tcgen05.mma consumes directly.
// * warp roles: warp 0 TMA producer, warp 1 MMA issuer (one elected thread), warp 2 TMEM allocator,
//   warps 4..11 epilogue.  smem ring of kStages, mbarrier full/empty pairs, one tcgen05.commit per stage.
// * an optional second accumulator (TMEM columns N..2N) receives the 1x1 shortcut conv of a ResidualBlock.
// * epilogue: thread = one output row (TMEM lane); GroupNorm statistics = in-thread sum over the group's columns +
//   warp-shuffle reduction over the L lanes of the trajectory; then GN-affine, Mish, FiLM, residual, bf16/fp32 store.
//
// Algorithmic HBM bytes per launch: 2*(batch*L*C_in + batch*L*C_out) (+ shortcut input), weights once through L2.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>

#include <cstdio>
#include <cstdlib>
#include <type_traits>

#include "common.cuh"
#include "ptx_sm100.cuh"

namespace cds {

constexpr int kTcThreads = 320;   // warps 0-7 epilogue (TMEM lane quarter = warp % 4, column slice = warp / 4),
                                  // warp 8 TMA producer, warp 9 TMEM allocator + MMA issuer
constexpr int kTcEpiThreads = 256;
constexpr int kTcMaxStages = 10;

struct ConvTcParams {
  CUtensorMap tm_a, tm_b, tm_a2, tm_b2;
  // output as a TMA-store target: box {16 channels, L positions, 32/L trajectories} = the 32 tile rows one epilogue warp owns
  // x 16 columns, staged in shared memory (SWIZZLE_64B for 4-byte / SWIZZLE_32B for 2-byte elements).  Valid when out_tma != 0.
  CUtensorMap tm_out;
  int out_tma;
  // SPLIT > 1 kernels: the SPLIT column-tile CTAs of a row tile form a thread-block cluster (cluster = SPLIT, else 1) and share
  // the activation tiles: CTA r fetches trajectories [r*T/SPLIT, (r+1)*T/SPLIT) of the tile (tm_a_mc / tm_a2_mc: the same
  // tensors with that smaller box) and MULTICASTS them into every CTA's stage -- the A bytes cross the L2 -> SM fabric once per
  // row tile instead of once per column tile.
  CUtensorMap tm_a_mc, tm_a2_mc;
  int cluster;
  // identity residual as a TMA-load source with the box of tm_out: the fast lane prefetches the next 32 rows x 16 columns of the
  // residual into per-warp staging rows while it works on the current ones (valid when res_tma != 0; tiles of N <= 64 only)
  CUtensorMap tm_res;
  int res_tma;
  int batch, L, log2L, C_out, taps, pad;   // L = output positions per tile-trajectory; C_out = channels per phase
  int num_tiles;                  // ceil(batch*L / 128); CTAs are persistent and stride over the tiles
  int phases;                     // 2: columns [0,C_out) / [C_out,2C_out) are output positions 2l / 2l+1 (transposed conv)
  int kchunks, kchunks2;          // channel chunks of the main conv / of the shortcut conv
  int in_batch_mod;
  int n_col_tiles;                // SPLIT == 1 kernels, no GroupNorm: the layer's columns as this many N-wide tiles (runtime)
  int sample_div;                 // per-trajectory vectors are indexed by (row's batch index) / sample_div   (>= 1)
  cds_vec bias, scale, shift;
  int groups; const float* gn_gamma; const float* gn_beta; float gn_eps;
  int act;
  const void* res; int64_t res_bstride; int res_lstride; int res_batch_mod; int res_dtype;
  const float* res_bias;
  void* out; int64_t out_bstride; int out_lstride; int out_dtype;
  long long* trace;               // debug: per-CTA clock64 timeline (kTraceSlots entries per CTA), normally NULL
};
constexpr int kTraceSlots = 64;
// [0] globaltimer at entry  [1] clock at entry  [2] clock after the prologue barrier  [3] clock at exit  [4] globaltimer at exit
// [5] tiles done by this CTA;  tile t (t < 14): [8+4t] producer issued its last k-block, [9+4t] MMA saw its first operands,
// [10+4t] epilogue saw the accumulator, [11+4t] epilogue done
__device__ __forceinline__ long long gtimer() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define CDS_TRACE(slot, val) do { if (p.trace) p.trace[(int64_t)blockIdx.x * kTraceSlots + (slot)] = (val); } while (0)

// MUFU approximations with flush-to-zero: ONE instruction each (the non-ftz forms expand into range fix-ups)
__device__ __forceinline__ float ex2_ftz(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_ftz(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rsqrt_ftz(float x) { float y; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// mish(y) + add as 7 issue slots:  tanh(softplus(y)) = 1 - 2 / (e^2 + 2e + 2),  e = exp(y).
// e = inf (y > 88) gives 1 - 2/inf = 1, i.e. mish(y) = y, which is torch's softplus-threshold behaviour; no clamp needed.
__device__ __forceinline__ float mish_fma(float y, float add) {
  const float e = ex2_ftz(y * 1.4426950408889634f);
  const float d = fmaf(e, e + 2.f, 2.f);
  const float w = fmaf(-2.f, rcp_ftz(d), 1.f);
  return fmaf(y, w, add);
}
__device__ __forceinline__ float fast_mish(float x) { return mish_fma(x, 0.f); }
__device__ __forceinline__ float fast_sigmoid(float x) { return rcp_ftz(1.f + ex2_ftz(-1.4426950408889634f * x)); }
// ACT is a compile-time constant inside the unrolled epilogue loops (a runtime switch there multiplies the code size
// by the number of activations and thrashes the instruction cache); kActOther keeps the generic runtime switch.
constexpr int kActOther = -1;
template <int ACT>
__device__ __forceinline__ float tc_act(int act, float x) {
  if constexpr (ACT == CDS_ACT_NONE) return x;
  else if constexpr (ACT == CDS_ACT_MISH) return fast_mish(x);
  else if constexpr (ACT == CDS_ACT_GELU_TANH) {          // 0.5 x (1 + tanh(u)) = x sigmoid(2u), u = sqrt(2/pi) (x + 0.044715 x^3)
    const float u = 0.7978845608028654f * (x + 0.044715f * x * x * x);
    return x * fast_sigmoid(2.f * u);
  }
  else {
    switch (act) {
      case CDS_ACT_MISH: return fast_mish(x);
      case CDS_ACT_SILU: return x * fast_sigmoid(x);
      case CDS_ACT_GELU_TANH: { float u = 0.7978845608028654f * (x + 0.044715f * x * x * x);   // 0.5 (1 + tanh(u)) = sigmoid(2u)
                                return x * fast_sigmoid(2.f * u); }
      case CDS_ACT_MISH_SILU: { float m = fast_mish(x); return m * fast_sigmoid(m); }
      case CDS_ACT_LEAKY_RELU: return x > 0.f ? x : 0.01f * x;
      case CDS_ACT_GELU_ERF: return 0.5f * x * (1.f + erff(x * 0.7071067811865476f));
      default: return x;
    }
  }
}

// GroupNorm coefficients of GPC groups from per-thread partial sums: all-reduce (s1, s2) over the L lanes that hold the
// trajectory's positions (lane groups of L consecutive lanes), return a = rstd and c = -mean * rstd per group so that
// (v - mean) * rstd = fma(v, a, c).  With V = 2 GPC >= 4 values the butterfly is "transposed": every round halves the
// number of values a lane carries (reduce-scatter), the survivors finish with log2(L / V) plain rounds, the lanes that
// end up with S1 and S2 of the same group swap them, compute (a, c), and V indexed shuffles hand every lane all groups:
// 2 V + log2(L / V) shuffles instead of V log2(L).
template <int GPC>
__device__ __forceinline__ void gn_coeffs(float (&s1)[GPC], float (&s2)[GPC], int L, int log2L, int lane, float inv_cnt,
                                          float eps, float (&a)[GPC], float (&c)[GPC]) {
  constexpr int V = 2 * GPC;
  constexpr unsigned kFull = 0xffffffffu;
  if (GPC >= 2 && L >= V) {
    float x[V];
#pragma unroll
    for (int g = 0; g < GPC; ++g) { x[g] = s1[g]; x[GPC + g] = s2[g]; }
    int off = L >> 1, log2V = 0;
#pragma unroll
    for (int half = V / 2; half >= 1; half >>= 1, off >>= 1, ++log2V) {
      const bool up = (lane & off) != 0;
#pragma unroll
      for (int i = 0; i < half; ++i) {
        const float send = up ? x[i] : x[i + half];
        const float keep = up ? x[i + half] : x[i];
        x[i] = keep + __shfl_xor_sync(kFull, send, off);
      }
    }
    for (; off >= 1; off >>= 1) x[0] += __shfl_xor_sync(kFull, x[0], off);
    const float other = __shfl_xor_sync(kFull, x[0], L >> 1);
    const bool st = (lane & (L >> 1)) != 0;
    const float S1 = st ? other : x[0], S2 = st ? x[0] : other;
    const float mean = S1 * inv_cnt;
    const float rstd = rsqrt_ftz(fmaxf(fmaf(S2, inv_cnt, -mean * mean), 0.f) + eps);
    const float av = rstd, cv = -mean * rstd;
    const int base = lane & ~(L - 1), sh = log2L - log2V;
#pragma unroll
    for (int g = 0; g < GPC; ++g) {
      a[g] = __shfl_sync(kFull, av, base | (g << sh));
      c[g] = __shfl_sync(kFull, cv, base | (g << sh));
    }
  } else {
    for (int off = L >> 1; off >= 1; off >>= 1) {
#pragma unroll
      for (int g = 0; g < GPC; ++g) {
        s1[g] += __shfl_xor_sync(kFull, s1[g], off);
        s2[g] += __shfl_xor_sync(kFull, s2[g], off);
      }
    }
#pragma unroll
    for (int g = 0; g < GPC; ++g) {
      const float mean = s1[g] * inv_cnt;
      const float rstd = rsqrt_ftz(fmaxf(fmaf(s2[g], inv_cnt, -mean * mean), 0.f) + eps);
      a[g] = rstd; c[g] = -mean * rstd;
    }
  }
}

// N = columns of one CTA tile; SPLIT = 2 when the layer's C_out = 2N columns are shared by two CTAs (more CTAs in flight for
// the deep, narrow-batch layers: L = 4 / 8 have only 128 / 256 row tiles), each owning 4 of the 8 GroupNorm groups.
template <int KC, int N, bool HAS_RES, int SPLIT = 1>
struct ConvTcCfg {
  static constexpr int kRowBytes = KC * 2;
  static constexpr int kABytes = 128 * kRowBytes;
  static constexpr int kBBytes = N * kRowBytes;
  static constexpr int kStageBytes = kABytes + kBBytes;
  // Operand ring: as deep as the shared memory of the designed residency allows (2 CTAs/SM: ~100 KB each; 1 CTA/SM: ~200 KB),
  // at least 3, at most kTcMaxStages.  A tile is taps x C_in/KC k-blocks (5..20): only a ring that holds more than one tile
  // lets the TMA producer run ahead of the tile whose accumulator the epilogue is still draining -- with 4 stages and
  // 5 k-blocks per tile every tile paid one exposed L2 round trip (~1 us) on the narrow layers.
  // (2 CTAs/SM: 227 KB - 2 x (22 KB static: per-column constants, 16 KB of epilogue store staging, barriers; + 16 KB of residual
  // staging for the narrow tiles) - 2 x 1 KB reserved)
  static constexpr bool kResStage = N <= 64;             // per-warp staging of TMA-prefetched identity residuals
  static constexpr int kRingBudget = (N <= 64 ? 72 : (N <= 128 ? 88 : 184)) * 1024;
  static constexpr int kStagesFit = kRingBudget / kStageBytes;
  static constexpr int kStages = kStagesFit < 3 ? 3 : (kStagesFit > kTcMaxStages ? kTcMaxStages : kStagesFit);
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024;
  static constexpr int kCols = N * SPLIT;                                 // columns of the whole layer
  static constexpr int kColsPerTile = N * (HAS_RES ? 2 : 1);             // main (+ shortcut) accumulator
  static constexpr int kAccBufs = 2 * kColsPerTile <= 512 ? 2 : 1;       // double-buffered when TMEM allows
  static constexpr uint32_t kTmemNeed = (uint32_t)(kAccBufs * kColsPerTile);
  static constexpr uint32_t kTmemCols = kTmemNeed <= 32 ? 32 : (kTmemNeed <= 64 ? 64 : (kTmemNeed <= 128 ? 128 : (kTmemNeed <= 256 ? 256 : 512)));   // power of two
  // GroupNorm lanes exist for the power-of-two tile widths only (the 160 / 192-wide tiles serve un-normalised Linear layers)
  static constexpr bool kGnOk = (N & (N - 1)) == 0;
  static constexpr int kEpiSplit = N >= 32 ? 2 : 1;     // epilogue warps per TMEM lane quarter (column split)
  // designed CTAs per SM: 2 (102 registers per thread: the epilogue keeps 16-32 columns live).  3 CTAs (68 registers) were
  // measured on the narrow tiles: the spills cost more than the extra residency buys (471 -> 490 us per iteration).
  static constexpr int kMinBlocks = N <= 128 ? 2 : 1;
};

// W consecutive activations (bf16 or fp32) <-> registers, 8/16-byte vector accesses
template <int W>
__device__ __forceinline__ void load_row(const void* base, int64_t off, int dtype, float (&r)[W]) {
  if (dtype == CDS_BF16) {
    const __nv_bfloat16* p = reinterpret_cast<const __nv_bfloat16*>(base) + off;
    if constexpr (W == 4) {
      uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
      float2 a = __bfloat1622float2(h[0]), b = __bfloat1622float2(h[1]);
      r[0] = a.x; r[1] = a.y; r[2] = b.x; r[3] = b.y;
    } else {
#pragma unroll
      for (int k = 0; k < W / 8; ++k) {
        uint4 u = __ldg(reinterpret_cast<const uint4*>(p) + k);
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
        for (int j = 0; j < 4; ++j) { float2 f = __bfloat1622float2(h[j]); r[8 * k + 2 * j] = f.x; r[8 * k + 2 * j + 1] = f.y; }
      }
    }
  } else {
    const float4* p = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + off);
#pragma unroll
    for (int k = 0; k < W / 4; ++k) { float4 f = __ldg(p + k); r[4 * k] = f.x; r[4 * k + 1] = f.y; r[4 * k + 2] = f.z; r[4 * k + 3] = f.w; }
  }
}
template <int W>
__device__ __forceinline__ void store_row(void* base, int64_t off, int dtype, const float (&v)[W]) {
  if (dtype == CDS_BF16) {
    __nv_bfloat16* p = reinterpret_cast<__nv_bfloat16*>(base) + off;
    if constexpr (W == 4) {
      uint2 u;
      __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
      h[0] = __floats2bfloat162_rn(v[0], v[1]); h[1] = __floats2bfloat162_rn(v[2], v[3]);
      *reinterpret_cast<uint2*>(p) = u;
    } else {
#pragma unroll
      for (int k = 0; k < W / 8; ++k) {
        uint4 u;
        __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
        for (int j = 0; j < 4; ++j) h[j] = __floats2bfloat162_rn(v[8 * k + 2 * j], v[8 * k + 2 * j + 1]);
        reinterpret_cast<uint4*>(p)[k] = u;
      }
    }
  } else if (dtype == CDS_TF32) {
    float4* p = reinterpret_cast<float4*>(reinterpret_cast<float*>(base) + off);
#pragma unroll
    for (int k = 0; k < W / 4; ++k)
      p[k] = make_float4(round_tf32(v[4 * k]), round_tf32(v[4 * k + 1]), round_tf32(v[4 * k + 2]), round_tf32(v[4 * k + 3]));
  } else {
    float4* p = reinterpret_cast<float4*>(reinterpret_cast<float*>(base) + off);
#pragma unroll
    for (int k = 0; k < W / 4; ++k) p[k] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
  }
}

template <int KC, int N, bool HAS_RES, int SPLIT, bool TF32>
__global__ void __launch_bounds__(kTcThreads, ConvTcCfg<KC, N, HAS_RES, SPLIT>::kMinBlocks)
conv_tc_kernel(const __grid_constant__ ConvTcParams p, const int* __restrict__ iter_ptr) {
  using Cfg = ConvTcCfg<KC, N, HAS_RES, SPLIT>;
  constexpr int kTcStages = Cfg::kStages;
  constexpr int KE = TF32 ? KC / 2 : KC;            // channels per chunk (elements along K of one operand row)
  // the fast lanes write the mode's activation dtype (TF32 kernels: fp32 storage rounded to TF32, CDS_TF32) and read residuals
  // of the same storage type (CDS_F32 and CDS_TF32 read alike)
  constexpr int kActDtype = TF32 ? CDS_TF32 : CDS_BF16;
  auto act_readable = [](int dt) { return TF32 ? (dt != CDS_BF16) : (dt == CDS_BF16); };
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[kTcMaxStages];
  __shared__ __align__(8) uint64_t empty_bar[kTcMaxStages];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];    // MMA -> epilogue, per accumulator buffer
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];   // epilogue -> MMA
  __shared__ uint32_t tmem_base_holder;
  // per-column constants of the epilogue, staged once per CTA while the main loop runs:
  // 0 bias  1 GN gamma  2 GN beta  3 FiLM scale  4 FiLM shift  5 shortcut bias   (iteration-indexed "step" parts)
  __shared__ __align__(16) float s_col[6][Cfg::kCols];
  // epilogue store staging: every epilogue warp owns 32 rows x 16 columns (2 KB of fp32 / 1 KB of bf16), written in the
  // swizzle of p.tm_out and handed to the TMA unit as one bulk store -- a warp-level st.global of its 32 rows would touch 32
  // different cache lines per instruction (measured: the LSU serialises them, the store's source registers stay locked and the
  // epilogue stalls on them), the bulk store writes whole sectors and costs the warp 4 conflict-free st.shared
  __shared__ __align__(1024) uint8_t s_stage[kTcEpiThreads / 32][2048];
  __shared__ __align__(1024) uint8_t s_resb[Cfg::kResStage ? kTcEpiThreads / 32 : 1][Cfg::kResStage ? 2048 : 16];
  __shared__ __align__(8) uint64_t res_bar[kTcEpiThreads / 32];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // operand ring, 1024-byte aligned (swizzle atoms)
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - ptx::smem_u32(smem_raw));

  const int T = 128 >> p.log2L;                       // trajectories per tile
  if (threadIdx.x == 0) { CDS_TRACE(0, gtimer()); CDS_TRACE(1, clock64()); }
  const int n_kb_main = p.taps * p.kchunks;
  const int n_kb = n_kb_main + (HAS_RES ? p.kchunks2 : 0);

  const int cs = SPLIT > 1 ? p.cluster : 1;           // cluster size (1 = no multicast)
  const uint32_t crank = cs > 1 ? ptx::cluster_ctarank() : 0u;
  const uint16_t cmask = (uint16_t)((1u << cs) - 1u);
  if (threadIdx.x == 0) {
    // a stage is free again when the MMAs of EVERY CTA of the cluster have consumed it (peers multicast into it)
    for (int s = 0; s < kTcStages; ++s) { ptx::mbar_init(&full_bar[s], 1); ptx::mbar_init(&empty_bar[s], (uint32_t)cs); }
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(&tmem_full_bar[i], 1); ptx::mbar_init(&tmem_empty_bar[i], kTcEpiThreads / 32); }
    for (int i = 0; i < kTcEpiThreads / 32; ++i) ptx::mbar_init(&res_bar[i], 1);
    ptx::fence_barrier_init();
  }
  if (warp == 8 && lane == 0) {
    ptx::prefetch_tensormap(&p.tm_a);
    ptx::prefetch_tensormap(&p.tm_b);
    if (HAS_RES) { ptx::prefetch_tensormap(&p.tm_a2); ptx::prefetch_tensormap(&p.tm_b2); }
    if (p.out_tma) ptx::prefetch_tensormap(&p.tm_out);
    if (cs > 1) { ptx::prefetch_tensormap(&p.tm_a_mc); if (HAS_RES) ptx::prefetch_tensormap(&p.tm_a2_mc); }
    if (p.res_tma) ptx::prefetch_tensormap(&p.tm_res);
  }
  if (warp == 9) ptx::tmem_alloc<Cfg::kTmemCols>(&tmem_base_holder);
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (cs > 1) ptx::cluster_sync();                    // every CTA's barriers exist before a peer can signal them
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = tmem_base_holder;
  if (threadIdx.x == 0) CDS_TRACE(2, clock64());
  // programmatic dependent launch: the next kernel of the stream may start its own prologue and weight prefetch now; it
  // blocks in grid_dep_wait() until this grid has completed before it touches anything a predecessor wrote
  if (threadIdx.x == 0) ptx::grid_dep_launch_dependents();

  if (warp == 8) {
    // ===================================== TMA producer =====================================
    if (ptx::elect_one()) {
      // Weights do not depend on the previous kernel: arm the first ring fill and fetch its W tiles BEFORE waiting for the
      // predecessor grid (programmatic dependent launch); the activation tiles of those stages follow after the wait.
      int pre = 0;
      if (blockIdx.x < p.num_tiles) {
        const int n_off0 = (int)(blockIdx.x % (SPLIT > 1 ? SPLIT : p.n_col_tiles)) * N;
        pre = n_kb < kTcStages ? n_kb : kTcStages;
        for (int kb = 0; kb < pre; ++kb) {
          uint8_t* sb = smem_al + kb * Cfg::kStageBytes + Cfg::kABytes;
          ptx::mbar_expect_tx(&full_bar[kb], Cfg::kStageBytes);
          if (!HAS_RES || kb < n_kb_main) {
            const int tap = kb / p.kchunks, ck = kb - tap * p.kchunks;
            ptx::tma_load_2d(sb, &p.tm_b, &full_bar[kb], ck * KE, tap * p.C_out * p.phases + n_off0);
          } else {
            ptx::tma_load_2d(sb, &p.tm_b2, &full_bar[kb], (kb - n_kb_main) * KE, n_off0);
          }
        }
      }
      ptx::grid_dep_wait();
      int ring = 0;                                   // k-blocks issued so far (smem ring position, across tiles)
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const int nct = SPLIT > 1 ? SPLIT : p.n_col_tiles;
      const int b0 = (tile / nct) * T;
      const int n_off = (tile % nct) * N;             // first layer column of this CTA tile
      const int a_b0 = p.in_batch_mod > 0 ? b0 % p.in_batch_mod : b0;
      const int r_b0 = p.res_batch_mod > 0 ? b0 % p.res_batch_mod : b0;
      for (int kb = 0; kb < n_kb; ++kb, ++ring) {
        const int s = ring % kTcStages;
        const uint32_t ph = (ring / kTcStages) & 1;
        const bool w_done = ring < pre;               // this stage was armed and its W tile fetched before the wait
        if (!w_done) {
          ptx::mbar_wait(&empty_bar[s], ph ^ 1);
          ptx::mbar_expect_tx(&full_bar[s], Cfg::kStageBytes);
        }
        uint8_t* sa = smem_al + s * Cfg::kStageBytes;
        uint8_t* sb = sa + Cfg::kABytes;
        if (!HAS_RES || kb < n_kb_main) {
          const int tap = kb / p.kchunks, ck = kb - tap * p.kchunks;
          if (cs == 1) ptx::tma_load_3d(sa, &p.tm_a, &full_bar[s], ck * KE, tap - p.pad, a_b0);
          else ptx::tma_load_3d_mc(sa + crank * (Cfg::kABytes / SPLIT), &p.tm_a_mc, &full_bar[s], ck * KE, tap - p.pad,
                                   a_b0 + (int)crank * (T / SPLIT), cmask);
          if (!w_done) ptx::tma_load_2d(sb, &p.tm_b, &full_bar[s], ck * KE, tap * p.C_out * p.phases + n_off);
        } else {
          const int ck = kb - n_kb_main;
          if (cs == 1) ptx::tma_load_3d(sa, &p.tm_a2, &full_bar[s], ck * KE, 0, r_b0);
          else ptx::tma_load_3d_mc(sa + crank * (Cfg::kABytes / SPLIT), &p.tm_a2_mc, &full_bar[s], ck * KE, 0,
                                   r_b0 + (int)crank * (T / SPLIT), cmask);
          if (!w_done) ptx::tma_load_2d(sb, &p.tm_b2, &full_bar[s], ck * KE, n_off);
        }
      }
      { const int t_i = (tile - blockIdx.x) / gridDim.x; if (t_i < 14) CDS_TRACE(8 + 4 * t_i, clock64()); }
      }
    }
  } else if (warp == 9) {
    // ===================================== MMA issuer =====================================
    if (ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc<TF32>(128, N);
      int ring = 0, it = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int buf = it % Cfg::kAccBufs;
      const uint32_t use = (uint32_t)(it / Cfg::kAccBufs);            // how often this buffer has been used before
      ptx::mbar_wait(&tmem_empty_bar[buf], (use & 1) ^ 1);              // epilogue has drained the previous use
      ptx::tc_fence_after_sync();
      const uint32_t acc_base = tmem_base + (uint32_t)(buf * Cfg::kColsPerTile);
      for (int kb = 0; kb < n_kb; ++kb, ++ring) {
        const int s = ring % kTcStages;
        const uint32_t ph = (ring / kTcStages) & 1;
        ptx::mbar_wait(&full_bar[s], ph);
        ptx::tc_fence_after_sync();
        if (kb == 0 && it < 14) CDS_TRACE(9 + 4 * it, clock64());
        const uint32_t sa = smem_base + s * Cfg::kStageBytes;
        const uint64_t da = ptx::make_kmajor_desc<Cfg::kRowBytes>(sa);
        const uint64_t db = ptx::make_kmajor_desc<Cfg::kRowBytes>(sa + Cfg::kABytes);
        const bool second = HAS_RES && kb >= n_kb_main;
        const uint32_t d_addr = acc_base + (second ? (uint32_t)N : 0u);
        const bool first_of_acc = second ? (kb == n_kb_main) : (kb == 0);
#pragma unroll
        for (int k = 0; k < KC / 16; ++k) {
          // advancing 16 bf16 / 8 tf32 (32 B) along K inside the swizzle span = +2 in the (addr >> 4) field
          ptx::umma<TF32>(d_addr, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (first_of_acc && k == 0) ? 0u : 1u);
        }
        // frees the smem slot once these MMAs have read it (in every CTA of the cluster when the slot is filled by multicast)
        if (cs > 1) ptx::umma_commit_mc(&empty_bar[s], cmask); else ptx::umma_commit(&empty_bar[s]);
      }
      ptx::umma_commit(&tmem_full_bar[buf]);      // this tile's accumulators complete
      }
    }
  } else {
    // ===================================== epilogue (warps 0..7) =====================================
    // thread = one output row (TMEM lane m) x NH columns.  Everything per ELEMENT is branch-free: the operator's options
    // pick one of a few compile-time specialised chunk loops (CTA-uniform dispatch, once per tile).
    ptx::grid_dep_wait();                           // iteration counter, tables, residual inputs: all written by predecessors
    const int iter = iter_ptr ? *iter_ptr : 0;
    constexpr int EW = Cfg::kEpiSplit;
    constexpr int NH = N / EW;                      // columns per thread
    const int q = warp & 3;                         // TMEM lane quarter this warp may touch
    const int half = warp >> 2;                     // which slice of the N columns this warp handles
    const bool active = half < EW;                  // warp-uniform (N = 16: only warps 0..3 work)
    const int n_real = p.C_out * p.phases;          // < N only for narrow heads (C_out <= 16)

    // ---- stage the per-column constants (overlaps with the TMA/MMA main loop): columns [first, first + kCols) of the layer
    auto stage_cols = [&](int first) {
      const float* bstep = p.bias.step ? p.bias.step + (int64_t)iter * p.bias.step_stride : nullptr;
      const float* sstep = p.scale.step ? p.scale.step + (int64_t)iter * p.scale.step_stride : nullptr;
      const float* hstep = p.shift.step ? p.shift.step + (int64_t)iter * p.shift.step_stride : nullptr;
      const bool scale_any = p.scale.step || p.scale.sample;
      const int cpg = p.groups > 0 ? p.C_out / p.groups : 0;
      for (int n = threadIdx.x; n < Cfg::kCols; n += kTcEpiThreads) {
        const bool real = first + n < n_real;
        const int c = real ? (first + n) % p.C_out : 0;
        s_col[0][n] = (real && bstep) ? __ldg(bstep + c) - (cpg ? group_mean(bstep, c - c % cpg, cpg) : 0.f) : 0.f;
        s_col[1][n] = (real && p.groups > 0) ? __ldg(p.gn_gamma + c) : 1.f;
        s_col[2][n] = (real && p.groups > 0) ? __ldg(p.gn_beta + c) : 0.f;
        s_col[3][n] = sstep ? (real ? __ldg(sstep + c) : 0.f) : (scale_any ? 0.f : 1.f);
        s_col[4][n] = (real && hstep) ? __ldg(hstep + c) : 0.f;
        s_col[5][n] = (real && HAS_RES && p.res_bias) ? __ldg(p.res_bias + c) : 0.f;
      }
    };
    stage_cols(0);
    ptx::named_bar_sync(1, kTcEpiThreads);

    // CTA-uniform option flags
    const bool has_gn = p.groups > 0;
    const bool smp = p.bias.sample || p.scale.sample || p.shift.sample;
    const bool has_scale = p.scale.step || p.scale.sample;
    const bool has_shift = p.shift.step || p.shift.sample;
    const bool io_vec = n_real == Cfg::kCols * (SPLIT > 1 ? 1 : p.n_col_tiles);     // every column of every tile is a real channel
    const bool add_res = p.res != nullptr;
    const int film = (smp || has_scale) ? 2 : (has_shift ? 1 : 0);

    const int m = 32 * q + lane;
    const int col0 = half * NH;
    int it = 0;

    // ---- fast lane: the UNet block conv (GroupNorm + Mish, optional additive time row, optional identity residual / shortcut
    // accumulator, bf16 in and out, every column real).  The narrow tiles run close to the ISSUE limit (4 epilogue warps per
    // scheduler at ~0.2 IPC each), so instructions per tile are what counts: the option dispatch happens ONCE per kernel (the
    // tile loop lives inside the specialisation), addresses are strength-reduced to one multiply-add per tile, dtypes are fixed.
    const bool fast_ok = N >= 32 && p.n_col_tiles <= 1 && has_gn && p.act == CDS_ACT_MISH && film != 2 && p.phases == 1 && io_vec &&
                         p.out_dtype == kActDtype && (!add_res || act_readable(p.res_dtype)) && p.res_batch_mod == 0 && p.out_tma;
    auto fast_tiles = [&](auto film_tag, auto res_tag) {
      constexpr bool SHIFT = decltype(film_tag)::value == 1;
      constexpr bool RES = decltype(res_tag)::value;
      constexpr int CPG = Cfg::kCols / 8;
      constexpr int WC = CPG > 16 ? CPG : 16;
      constexpr int GPC = WC / CPG;
      const int T_ = 128 >> p.log2L;
      const int tb = m >> p.log2L, l = m & (p.L - 1);              // trajectory inside the tile / position: tile-invariant
      const float inv_cnt = 1.f / (float)(p.L * CPG);
      const float eps = p.gn_eps;
      const int L_ = p.L, log2L_ = p.log2L, batch_ = p.batch;
      using ET = std::conditional_t<TF32, float, __nv_bfloat16>;     // activation element
      const ET* const res_l = RES ? reinterpret_cast<const ET*>(p.res) + (int64_t)l * p.res_lstride : nullptr;
      uint8_t* const stg = &s_stage[warp][0];                         // this warp's 32 rows x 16 columns
      uint8_t* const stg_row = stg + lane * (16 * (int)sizeof(ET));
      const int traj_q = (32 * q) >> p.log2L;                         // first trajectory of this warp's rows inside the tile
      const int64_t res_bs = p.res_bstride;
      // identity residual through TMA: this warp's 32 rows x 16 columns of the NEXT column group / tile are fetched into its
      // staging rows while the current group is processed (the strided ld.global of a row-per-thread layout cost ~1 us per tile)
      constexpr int kGroups = NH / 16;                                // 16-column groups per thread and tile
      constexpr uint32_t kResBytes = 32u * 16u * (uint32_t)sizeof(ET);
      const bool res_pf = RES && Cfg::kResStage && p.res_tma != 0;
      uint8_t* const rstg = &s_resb[Cfg::kResStage ? warp : 0][0];
      uint32_t res_phase = 0;
      auto issue_res = [&](int tile_, int gi_) {                      // lane 0 only
        ptx::mbar_expect_tx(&res_bar[warp], kResBytes);
        ptx::tma_load_3d(rstg, &p.tm_res, &res_bar[warp], (tile_ % SPLIT) * N + col0 + 16 * gi_, 0, (tile_ / SPLIT) * T_ + traj_q);
      };
      if (res_pf && lane == 0 && (int)blockIdx.x < p.num_tiles) issue_res((int)blockIdx.x, 0);
      const uint32_t t_lane = tmem_base + ((uint32_t)(32 * q) << 16);
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
        const int buf = it % Cfg::kAccBufs;
        const uint32_t use = (uint32_t)(it / Cfg::kAccBufs);
        const int n_off = (tile % SPLIT) * N;
        const int b = (tile / SPLIT) * T_ + tb;
        const bool valid = b < batch_;
        const uint32_t t_row = t_lane + (uint32_t)(buf * Cfg::kColsPerTile);
        const int traj0 = (tile / SPLIT) * T_ + traj_q;
        const ET* const res_row_p = RES ? res_l + (int64_t)b * res_bs + n_off : nullptr;
        ptx::mbar_wait(&tmem_full_bar[buf], use & 1);
        ptx::tc_fence_after_sync();
        if (threadIdx.x == 0 && it < 14) CDS_TRACE(10 + 4 * it, clock64());
#pragma unroll 1
        for (int ch = 0; ch < NH / WC; ++ch) {
          const int n0 = col0 + ch * WC;                            // CTA-tile column
          const float* const cb = &s_col[0][n_off + n0];            // staged constants of these columns (row stride kCols)
          float v[WC];
          ptx::tmem_ld<WC>(t_row + (uint32_t)n0, v);
          float s1[GPC], s2[GPC], ga[GPC], gc[GPC];
#pragma unroll
          for (int g = 0; g < GPC; ++g) { s1[g] = 0.f; s2[g] = 0.f; }
#pragma unroll
          for (int k = 0; k < WC / 4; ++k) {
            const float4 bb = reinterpret_cast<const float4*>(cb)[k];
            const int g = (4 * k) / CPG;
            const float x0 = (v[4 * k] += bb.x), x1 = (v[4 * k + 1] += bb.y), x2 = (v[4 * k + 2] += bb.z), x3 = (v[4 * k + 3] += bb.w);
            s1[g] += (x0 + x1) + (x2 + x3);
            s2[g] = fmaf(x0, x0, s2[g]); s2[g] = fmaf(x1, x1, s2[g]); s2[g] = fmaf(x2, x2, s2[g]); s2[g] = fmaf(x3, x3, s2[g]);
          }
          gn_coeffs<GPC>(s1, s2, L_, log2L_, lane, inv_cnt, eps, ga, gc);
#pragma unroll
          for (int h = 0; h < WC / 16; ++h) {
            float addv[16];
            if constexpr (SHIFT) {
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float4 sft = reinterpret_cast<const float4*>(cb + 4 * Cfg::kCols + 16 * h)[k];
                addv[4 * k] = sft.x; addv[4 * k + 1] = sft.y; addv[4 * k + 2] = sft.z; addv[4 * k + 3] = sft.w;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j) addv[j] = 0.f;
            }
            if (RES && res_pf) {
              // the prefetched rows (zero beyond the batch: TMA out-of-bound fill), de-swizzled like the store staging
              ptx::mbar_wait(&res_bar[warp], res_phase);
              res_phase ^= 1u;
              const uint8_t* rr = rstg + lane * (16 * (int)sizeof(ET));
              if constexpr (TF32) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const float4 rv = *reinterpret_cast<const float4*>(rr + ((k ^ ((lane >> 1) & 3)) << 4));
                  addv[4 * k] += rv.x; addv[4 * k + 1] += rv.y; addv[4 * k + 2] += rv.z; addv[4 * k + 3] += rv.w;
                }
              } else {
                const int sw = (lane >> 2) & 1;
                const uint4 u0 = *reinterpret_cast<const uint4*>(rr + ((0 ^ sw) << 4)), u1 = *reinterpret_cast<const uint4*>(rr + ((1 ^ sw) << 4));
                const uint32_t w[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  addv[2 * j] += __uint_as_float(w[j] << 16);
                  addv[2 * j + 1] += __uint_as_float(w[j] & 0xffff0000u);
                }
              }
              __syncwarp();                                          // every lane has its values: the rows may be overwritten
              if (lane == 0) {
                const int gi = ch * (WC / 16) + h;
                if (gi + 1 < kGroups) { ptx::fence_proxy_async(); issue_res(tile, gi + 1); }
                else if (tile + (int)gridDim.x < p.num_tiles) { ptx::fence_proxy_async(); issue_res(tile + (int)gridDim.x, 0); }
              }
            } else if constexpr (RES && TF32) {
              if (valid) {
                const float4* rp = reinterpret_cast<const float4*>(res_row_p + n0 + 16 * h);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const float4 rv = rp[k];
                  addv[4 * k] += rv.x; addv[4 * k + 1] += rv.y; addv[4 * k + 2] += rv.z; addv[4 * k + 3] += rv.w;
                }
              }
            } else if constexpr (RES) {
              uint4 u0 = make_uint4(0, 0, 0, 0), u1 = u0;
              if (valid) { const uint4* rp = reinterpret_cast<const uint4*>(res_row_p + n0 + 16 * h); u0 = rp[0]; u1 = rp[1]; }
              const uint32_t w[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
#pragma unroll
              for (int j = 0; j < 8; ++j) {                           // bf16 pair -> two fp32: shift / mask, no cvt
                addv[2 * j] += __uint_as_float(w[j] << 16);
                addv[2 * j + 1] += __uint_as_float(w[j] & 0xffff0000u);
              }
            }
            if constexpr (HAS_RES) {
              float r2[16];
              ptx::tmem_ld<16>(t_row + (uint32_t)(N + n0 + 16 * h), r2);
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float4 rb = reinterpret_cast<const float4*>(cb + 5 * Cfg::kCols + 16 * h)[k];
                addv[4 * k] += r2[4 * k] + rb.x; addv[4 * k + 1] += r2[4 * k + 1] + rb.y;
                addv[4 * k + 2] += r2[4 * k + 2] + rb.z; addv[4 * k + 3] += r2[4 * k + 3] + rb.w;
              }
            }
            uint32_t packed[8];
            // the warp's staging rows are free again once its previous bulk store has READ them
            if (lane == 0) ptx::bulk_wait_group_read<0>();
            __syncwarp();
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float4 gm = reinterpret_cast<const float4*>(cb + 1 * Cfg::kCols + 16 * h)[k];
              const float4 be = reinterpret_cast<const float4*>(cb + 2 * Cfg::kCols + 16 * h)[k];
              const int g = (16 * h + 4 * k) / CPG;
              const float o0 = mish_fma(fmaf(fmaf(v[16 * h + 4 * k + 0], ga[g], gc[g]), gm.x, be.x), addv[4 * k + 0]);
              const float o1 = mish_fma(fmaf(fmaf(v[16 * h + 4 * k + 1], ga[g], gc[g]), gm.y, be.y), addv[4 * k + 1]);
              const float o2 = mish_fma(fmaf(fmaf(v[16 * h + 4 * k + 2], ga[g], gc[g]), gm.z, be.z), addv[4 * k + 2]);
              const float o3 = mish_fma(fmaf(fmaf(v[16 * h + 4 * k + 3], ga[g], gc[g]), gm.w, be.w), addv[4 * k + 3]);
              if constexpr (TF32) {
                // 16-byte chunk k of this row's 64 staged bytes, SWIZZLE_64B: chunk index ^= address bits [7:8] = (row >> 1) & 3
                *reinterpret_cast<float4*>(stg_row + ((k ^ ((lane >> 1) & 3)) << 4)) =
                    make_float4(round_tf32(o0), round_tf32(o1), round_tf32(o2), round_tf32(o3));
              } else {
                __nv_bfloat162 p01 = __floats2bfloat162_rn(o0, o1), p23 = __floats2bfloat162_rn(o2, o3);
                packed[2 * k] = *reinterpret_cast<uint32_t*>(&p01);
                packed[2 * k + 1] = *reinterpret_cast<uint32_t*>(&p23);
              }
            }
            if constexpr (!TF32) {     // 32 staged bytes per row, SWIZZLE_32B: chunk index ^= address bit 7 = (row >> 2) & 1
              const int sw = (lane >> 2) & 1;
              *reinterpret_cast<uint4*>(stg_row + ((0 ^ sw) << 4)) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
              *reinterpret_cast<uint4*>(stg_row + ((1 ^ sw) << 4)) = make_uint4(packed[4], packed[5], packed[6], packed[7]);
            }
            ptx::fence_proxy_async();                       // generic-proxy writes -> visible to the TMA unit
            __syncwarp();
            if (lane == 0) {
              ptx::tma_store_3d(&p.tm_out, stg, n_off + n0 + 16 * h, 0, traj0);
              ptx::bulk_commit_group();
            }
          }
        }
        // hand the accumulator buffer back to the MMA warp (one arrival per epilogue warp)
        ptx::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&tmem_empty_bar[buf]);
        if (threadIdx.x == 0 && it < 14) CDS_TRACE(11 + 4 * it, clock64());
      }
    };
    if constexpr (N >= 32 && Cfg::kCols <= 256 && Cfg::kGnOk) {
      if (fast_ok) {
        using T1 = std::integral_constant<int, 1>;
        using T0 = std::integral_constant<int, 0>;
        if (film == 1) { if (add_res) fast_tiles(T1{}, std::true_type{}); else fast_tiles(T1{}, std::false_type{}); }
        else { if (add_res) fast_tiles(T0{}, std::true_type{}); else fast_tiles(T0{}, std::false_type{}); }
      }
    }
    // ---- plain lane: no GroupNorm, no FiLM, no residual -- bias + one activation + store (the resampling convs of the UNets,
    // DiT1d's QKV and GELU Linear layers).  Same idea as the fast lane: dispatch once, strength-reduced addressing, fixed dtype.
    const bool plain_ok = N >= 32 && !HAS_RES && !has_gn && film == 0 && !smp && !add_res && io_vec && p.res_batch_mod == 0 &&
                          (p.act == CDS_ACT_NONE || p.act == CDS_ACT_GELU_TANH);
    // ... and its "gated" form: out = (acc + bias) * gate(trajectory, column) + residual -- DiT1d's attention out-projection and
    // second MLP Linear (dit.py:33-36: x + gate * f(...)), fp32 residual stream, per-trajectory gate row
    const bool gated_ok = N >= 32 && !HAS_RES && !has_gn && p.act == CDS_ACT_NONE && p.scale.sample && !p.scale.step && !has_shift &&
                          !p.bias.sample && add_res && p.out_dtype != CDS_BF16 && io_vec && p.phases == 1 &&
                          p.res_batch_mod == 0 && p.out_tma == 1 && ((uintptr_t)p.scale.sample % 16 == 0) && (p.scale.sample_stride % 4 == 0);
    // ... and its "table" form: out = acc + bias + table[row % period] -- DiT1d's x_proj + pos_emb (dit.py:118), fp32 table
    const bool table_ok = N >= 32 && !HAS_RES && !has_gn && film == 0 && !smp && add_res && p.res_batch_mod > 0 && p.act == CDS_ACT_NONE &&
                          p.res_dtype != CDS_BF16 && p.out_dtype != CDS_BF16 && io_vec && p.phases == 1 && p.out_tma == 1 &&
                          ((uintptr_t)p.res % 16 == 0) && (p.res_bstride % 4 == 0) && (p.res_lstride % 4 == 0);
    auto plain_tiles = [&](auto act_tag, auto bf16_tag, auto mode_tag) {
      constexpr int ACT = decltype(act_tag)::value;
      constexpr int OUT_DT = decltype(bf16_tag)::value;            // cds_dtype of the output
      constexpr bool OUT_BF16 = OUT_DT == CDS_BF16;
      constexpr int MODE = decltype(mode_tag)::value;              // 0 plain, 1 gated + residual, 2 + periodic table
      constexpr bool GATED = MODE == 1;
      const int T_ = 128 >> p.log2L;
      const int tb = m >> p.log2L, l = m & (p.L - 1);
      const int nct = SPLIT > 1 ? SPLIT : p.n_col_tiles;
      const int batch_ = p.batch, phases_ = p.phases, C_out_ = p.C_out;
      const int64_t out_bs = p.out_bstride, out_ls = p.out_lstride;
      const uint32_t t_lane = tmem_base + ((uint32_t)(32 * q) << 16);
      // out_tma: 1 = {C, L, batch} view (one phase), 2 = {C, phase, L, batch} view of a two-phase transposed conv's output
      const int use_tma = p.out_tma;
      uint8_t* const stg = &s_stage[warp][0];
      const int traj_q = (32 * q) >> p.log2L;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
        const int buf = it % Cfg::kAccBufs;
        const uint32_t use = (uint32_t)(it / Cfg::kAccBufs);
        const int n_off = (tile % nct) * N;
        const int sc_off = SPLIT > 1 ? n_off : 0;
        if (SPLIT == 1 && nct > 1) {                   // runtime column tiles: this tile's constants
          ptx::named_bar_sync(1, kTcEpiThreads);
          stage_cols(n_off);
          ptx::named_bar_sync(1, kTcEpiThreads);
        }
        const int b = (tile / nct) * T_ + tb;
        const bool valid = b < batch_;
        const uint32_t t_row = t_lane + (uint32_t)(buf * Cfg::kColsPerTile);
        ptx::mbar_wait(&tmem_full_bar[buf], use & 1);
        ptx::tc_fence_after_sync();
        if (threadIdx.x == 0 && it < 14) CDS_TRACE(10 + 4 * it, clock64());
#pragma unroll 1
        for (int ch = 0; ch < NH / 16; ++ch) {
          const int n0 = col0 + ch * 16;
          const int ng0 = n_off + n0;                               // layer column (phase-major for transposed convs)
          const int phase = (phases_ == 1 || ng0 < C_out_) ? 0 : 1;
          const int c0 = ng0 - phase * C_out_;
          float v[16];
          ptx::tmem_ld<16>(t_row + (uint32_t)n0, v);
          const float4* b4 = reinterpret_cast<const float4*>(&s_col[0][sc_off + n0]);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float4 bb = b4[k];
            v[4 * k] = tc_act<ACT>(ACT, v[4 * k] + bb.x); v[4 * k + 1] = tc_act<ACT>(ACT, v[4 * k + 1] + bb.y);
            v[4 * k + 2] = tc_act<ACT>(ACT, v[4 * k + 2] + bb.z); v[4 * k + 3] = tc_act<ACT>(ACT, v[4 * k + 3] + bb.w);
          }
          if constexpr (GATED) {
            const int bs = p.sample_div > 1 ? b / p.sample_div : b;
            float4 g4[4], r4[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) { g4[k] = make_float4(0.f, 0.f, 0.f, 0.f); r4[k] = g4[k]; }
            if (valid) {
              const float4* gp = reinterpret_cast<const float4*>(p.scale.sample + (int64_t)bs * p.scale.sample_stride + c0);
              const int64_t ro = (int64_t)b * p.res_bstride + (int64_t)l * p.res_lstride + c0;
#pragma unroll
              for (int k = 0; k < 4; ++k) g4[k] = __ldg(gp + k);
              if (p.res_dtype == CDS_BF16) {           // (bf16 programs: the modulated tokens are bf16, the stream fp32)
                const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.res) + ro);
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                  const uint4 u = rp[k];
                  r4[2 * k] = make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                                          __uint_as_float(u.y & 0xffff0000u));
                  r4[2 * k + 1] = make_float4(__uint_as_float(u.z << 16), __uint_as_float(u.z & 0xffff0000u), __uint_as_float(u.w << 16),
                                              __uint_as_float(u.w & 0xffff0000u));
                }
              } else {
                const float4* rp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.res) + ro);
#pragma unroll
                for (int k = 0; k < 4; ++k) r4[k] = rp[k];
              }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              v[4 * k] = fmaf(v[4 * k], g4[k].x, r4[k].x); v[4 * k + 1] = fmaf(v[4 * k + 1], g4[k].y, r4[k].y);
              v[4 * k + 2] = fmaf(v[4 * k + 2], g4[k].z, r4[k].z); v[4 * k + 3] = fmaf(v[4 * k + 3], g4[k].w, r4[k].w);
            }
          }
          if constexpr (MODE == 2) {
            if (valid) {
              const float4* rp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.res) +
                                                                 (int64_t)(b % p.res_batch_mod) * p.res_bstride + (int64_t)l * p.res_lstride + c0);
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float4 r = __ldg(rp + k);
                v[4 * k] += r.x; v[4 * k + 1] += r.y; v[4 * k + 2] += r.z; v[4 * k + 3] += r.w;
              }
            }
          }
          if (use_tma) {
            // through the warp's staging rows and one bulk store (see s_stage); rows beyond the batch are clipped by the TMA unit
            if (lane == 0) ptx::bulk_wait_group_read<0>();
            __syncwarp();
            if constexpr (OUT_BF16) {
              uint32_t w[8];
#pragma unroll
              for (int k = 0; k < 8; ++k) { __nv_bfloat162 h2 = __floats2bfloat162_rn(v[2 * k], v[2 * k + 1]); w[k] = *reinterpret_cast<uint32_t*>(&h2); }
              uint8_t* const sr = stg + lane * 32;
              const int sw = (lane >> 2) & 1;
              *reinterpret_cast<uint4*>(sr + ((0 ^ sw) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
              *reinterpret_cast<uint4*>(sr + ((1 ^ sw) << 4)) = make_uint4(w[4], w[5], w[6], w[7]);
            } else {
              uint8_t* const sr = stg + lane * 64;
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                float4 o4;
                if constexpr (OUT_DT == CDS_TF32)
                  o4 = make_float4(round_tf32(v[4 * k]), round_tf32(v[4 * k + 1]), round_tf32(v[4 * k + 2]), round_tf32(v[4 * k + 3]));
                else o4 = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
                *reinterpret_cast<float4*>(sr + ((k ^ ((lane >> 1) & 3)) << 4)) = o4;
              }
            }
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              if (use_tma == 2) ptx::tma_store_4d(&p.tm_out, stg, c0, phase, 0, (tile / nct) * T_ + traj_q);
              else ptx::tma_store_3d(&p.tm_out, stg, c0, 0, (tile / nct) * T_ + traj_q);
              ptx::bulk_commit_group();
            }
          } else if (valid) {
            const int64_t oo = (int64_t)b * out_bs + (int64_t)(l * phases_ + phase) * out_ls + c0;
            if constexpr (OUT_BF16) {
              uint32_t w[8];
#pragma unroll
              for (int k = 0; k < 8; ++k) { __nv_bfloat162 h2 = __floats2bfloat162_rn(v[2 * k], v[2 * k + 1]); w[k] = *reinterpret_cast<uint32_t*>(&h2); }
              uint4* op = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + oo);
              op[0] = make_uint4(w[0], w[1], w[2], w[3]);
              op[1] = make_uint4(w[4], w[5], w[6], w[7]);
            } else {
              float4* op = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + oo);
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                if constexpr (OUT_DT == CDS_TF32)
                  op[k] = make_float4(round_tf32(v[4 * k]), round_tf32(v[4 * k + 1]), round_tf32(v[4 * k + 2]), round_tf32(v[4 * k + 3]));
                else op[k] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
              }
            }
          }
        }
        ptx::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&tmem_empty_bar[buf]);
        if (threadIdx.x == 0 && it < 14) CDS_TRACE(11 + 4 * it, clock64());
      }
    };
    if constexpr (N >= 32 && !HAS_RES) {
      using G = std::integral_constant<int, CDS_ACT_GELU_TANH>;
      using Z = std::integral_constant<int, CDS_ACT_NONE>;
      using DF = std::integral_constant<int, CDS_F32>;
      using DB = std::integral_constant<int, CDS_BF16>;
      using DT = std::integral_constant<int, CDS_TF32>;
      const int od = p.out_dtype;
      using M1 = std::integral_constant<int, 1>;
      using M2 = std::integral_constant<int, 2>;
      if (gated_ok && it == 0) {
        if (od == CDS_TF32) plain_tiles(Z{}, DT{}, M1{}); else plain_tiles(Z{}, DF{}, M1{});
      } else if (table_ok && it == 0) {
        if (od == CDS_TF32) plain_tiles(Z{}, DT{}, M2{}); else plain_tiles(Z{}, DF{}, M2{});
      } else if (plain_ok && it == 0) {
        using NG = std::integral_constant<int, 0>;
        if (p.act == CDS_ACT_GELU_TANH) {
          if (od == CDS_BF16) plain_tiles(G{}, DB{}, NG{}); else if (od == CDS_TF32) plain_tiles(G{}, DT{}, NG{}); else plain_tiles(G{}, DF{}, NG{});
        } else {
          if (od == CDS_BF16) plain_tiles(Z{}, DB{}, NG{}); else if (od == CDS_TF32) plain_tiles(Z{}, DT{}, NG{}); else plain_tiles(Z{}, DF{}, NG{});
        }
      }
    }
    // generic lane (everything else; a no-op after the fast lane: `it` then already counts all of this CTA's tiles)
    for (int tile = blockIdx.x + it * (int)gridDim.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
    const int buf = it % Cfg::kAccBufs;
    const uint32_t use = (uint32_t)(it / Cfg::kAccBufs);
    const int nct = SPLIT > 1 ? SPLIT : p.n_col_tiles;
    const int64_t row = (int64_t)(tile / nct) * 128 + m;
    const int n_off = (tile % nct) * N;
    // s_col holds the kCols = N*SPLIT columns of the layer; with runtime column tiles (SPLIT == 1, n_col_tiles > 1) it holds the
    // N columns of the CURRENT tile and is re-staged whenever the column tile changes
    const int sc_off = SPLIT > 1 ? n_off : 0;
    if (SPLIT == 1 && p.n_col_tiles > 1) {
      ptx::named_bar_sync(1, kTcEpiThreads);        // everybody has left the previous tile's constants
      stage_cols(n_off);
      ptx::named_bar_sync(1, kTcEpiThreads);
    }
    const bool valid = active && row < (int64_t)p.batch * p.L;
    const int b = (int)(row >> p.log2L), l = (int)(row & (p.L - 1));
    const uint32_t t_row = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(buf * Cfg::kColsPerTile);
    const int bs = p.sample_div > 1 ? b / p.sample_div : b;        // owner of the per-trajectory vectors (flattened token rows)
    const float* bias_smp = p.bias.sample ? p.bias.sample + (int64_t)bs * p.bias.sample_stride : nullptr;
    const float* scale_smp = p.scale.sample ? p.scale.sample + (int64_t)bs * p.scale.sample_stride : nullptr;
    const float* shift_smp = p.shift.sample ? p.shift.sample + (int64_t)bs * p.shift.sample_stride : nullptr;
    const int rb = p.res_batch_mod > 0 ? b % p.res_batch_mod : b;
    const int64_t res_row = (int64_t)rb * p.res_bstride + (int64_t)l * p.res_lstride;

    ptx::mbar_wait(&tmem_full_bar[buf], use & 1);
    ptx::tc_fence_after_sync();
    if (threadIdx.x == 0 && it < 14) CDS_TRACE(10 + 4 * it, clock64());

    // ---- 16 finished pre-activation columns (y) -> activation, FiLM, residual(s), store.  n0 = CTA-tile column.
    // FILM: 0 none, 1 additive per-iteration row (staged in smem), 2 anything (scale and/or per-trajectory rows)
    auto post16 = [&](auto act_tag, auto film_tag, auto& yv, auto off_tag, int n0) {
      constexpr int ACT = decltype(act_tag)::value;
      constexpr int FILM = decltype(film_tag)::value;
      constexpr int YO = decltype(off_tag)::value;                 // offset of these 16 columns inside yv[]
      const int ng0 = n_off + n0;                                 // layer column of the chunk's first element
      const int sg0 = sc_off + n0;                                // ... and where its constants sit in s_col
      const int phase = (p.phases == 1 || ng0 < p.C_out) ? 0 : 1;
      const int c0 = ng0 - phase * p.C_out;                       // its channel
      float addv[16];                                             // everything that is ADDED after the activation
      if constexpr (FILM == 1) {
        const float4* sh4 = reinterpret_cast<const float4*>(&s_col[4][sg0]);
#pragma unroll
        for (int k = 0; k < 4; ++k) { const float4 s = sh4[k]; addv[4 * k] = s.x; addv[4 * k + 1] = s.y; addv[4 * k + 2] = s.z; addv[4 * k + 3] = s.w; }
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) addv[j] = 0.f;
      }
      if (add_res) {
        float resv[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) resv[j] = 0.f;
        if (valid) load_row<16>(p.res, res_row + c0, p.res_dtype, resv);
#pragma unroll
        for (int j = 0; j < 16; ++j) addv[j] += resv[j];
      }
      if constexpr (HAS_RES) {
        float r2[16];
        ptx::tmem_ld<16>(t_row + (uint32_t)(N + n0), r2);
        const float4* rb4 = reinterpret_cast<const float4*>(&s_col[5][sg0]);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float4 s = rb4[k];
          addv[4 * k] += r2[4 * k] + s.x; addv[4 * k + 1] += r2[4 * k + 1] + s.y;
          addv[4 * k + 2] += r2[4 * k + 2] + s.z; addv[4 * k + 3] += r2[4 * k + 3] + s.w;
        }
      }
      float o[16];
      if constexpr (FILM == 2) {
        float sc[16], sh[16];
        const float4* sc4 = reinterpret_cast<const float4*>(&s_col[3][sg0]);
        const float4* sh4 = reinterpret_cast<const float4*>(&s_col[4][sg0]);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float4 a = sc4[k], d = sh4[k];
          sc[4 * k] = a.x; sc[4 * k + 1] = a.y; sc[4 * k + 2] = a.z; sc[4 * k + 3] = a.w;
          sh[4 * k] = d.x; sh[4 * k + 1] = d.y; sh[4 * k + 2] = d.z; sh[4 * k + 3] = d.w;
        }
        // per-trajectory FiLM rows: four 16-byte loads per vector when every column is a real channel and the rows are aligned
        // (ChiUNet1d: always), element-wise otherwise
        const bool film_vec = io_vec && (((uintptr_t)scale_smp | (uintptr_t)shift_smp) % 16 == 0);
        if (scale_smp && valid) {
          if (film_vec) {
            const float4* q4 = reinterpret_cast<const float4*>(scale_smp + c0);
#pragma unroll
            for (int k = 0; k < 4; ++k) { const float4 a = __ldg(q4 + k); sc[4 * k] += a.x; sc[4 * k + 1] += a.y; sc[4 * k + 2] += a.z; sc[4 * k + 3] += a.w; }
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) if (c0 + j < p.C_out) sc[j] += __ldg(scale_smp + c0 + j);
          }
        }
        if (shift_smp && valid) {
          if (film_vec) {
            const float4* q4 = reinterpret_cast<const float4*>(shift_smp + c0);
#pragma unroll
            for (int k = 0; k < 4; ++k) { const float4 a = __ldg(q4 + k); sh[4 * k] += a.x; sh[4 * k + 1] += a.y; sh[4 * k + 2] += a.z; sh[4 * k + 3] += a.w; }
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) if (c0 + j < p.C_out) sh[j] += __ldg(shift_smp + c0 + j);
          }
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) o[j] = fmaf(tc_act<ACT>(p.act, yv[YO + j]), sc[j], sh[j]) + addv[j];
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          if constexpr (ACT == CDS_ACT_MISH) o[j] = mish_fma(yv[YO + j], addv[j]);
          else o[j] = tc_act<ACT>(p.act, yv[YO + j]) + addv[j];
        }
      }
      if (p.out_tma == 1 && io_vec) {
        // like the fast / plain lanes: the warp's 32 rows x 16 columns through its swizzled staging rows and ONE bulk tensor store
        // (a thread storing its own row reaches a third of that: profiles/r02_micro_store_patterns.txt).  This is the lane of
        // ChiUNet1d's FiLM convs (per-trajectory scale and shift); rows beyond the batch are clipped by the TMA unit.
        uint8_t* const stg = &s_stage[warp][0];
        if (lane == 0) ptx::bulk_wait_group_read<0>();
        __syncwarp();
        if (p.out_dtype == CDS_BF16) {
          uint32_t w[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) { __nv_bfloat162 h2 = __floats2bfloat162_rn(o[2 * k], o[2 * k + 1]); w[k] = *reinterpret_cast<uint32_t*>(&h2); }
          uint8_t* const sr = stg + lane * 32;
          const int sw = (lane >> 2) & 1;
          *reinterpret_cast<uint4*>(sr + ((0 ^ sw) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
          *reinterpret_cast<uint4*>(sr + ((1 ^ sw) << 4)) = make_uint4(w[4], w[5], w[6], w[7]);
        } else {
          uint8_t* const sr = stg + lane * 64;
          const bool rnd = p.out_dtype == CDS_TF32;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float4 o4 = make_float4(o[4 * k], o[4 * k + 1], o[4 * k + 2], o[4 * k + 3]);
            if (rnd) o4 = make_float4(round_tf32(o4.x), round_tf32(o4.y), round_tf32(o4.z), round_tf32(o4.w));
            *reinterpret_cast<float4*>(sr + ((k ^ ((lane >> 1) & 3)) << 4)) = o4;
          }
        }
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          ptx::tma_store_3d(&p.tm_out, stg, c0, 0, (tile / nct) * (128 >> p.log2L) + ((32 * q) >> p.log2L));
          ptx::bulk_commit_group();
        }
        return;
      }
      if (!valid) return;
      const int64_t oo = (int64_t)b * p.out_bstride + (int64_t)(l * p.phases + phase) * p.out_lstride + c0;
      if (io_vec) {
        store_row<16>(p.out, oo, p.out_dtype, o);
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          if (c0 + j < p.C_out) {
            if (p.out_dtype == CDS_BF16) reinterpret_cast<__nv_bfloat16*>(p.out)[oo + j] = __float2bfloat16_rn(o[j]);
            else reinterpret_cast<float*>(p.out)[oo + j] = f32_for_store(o[j], p.out_dtype);
          }
        }
      }
    };

    // v[j] += bias(column) for WC columns starting at CTA-tile column n0 (float4 reads of the staged constants)
    auto add_bias = [&](auto wc_tag, auto& v, int n0) {
      constexpr int WC = decltype(wc_tag)::value;
      const float4* b4 = reinterpret_cast<const float4*>(&s_col[0][sc_off + n0]);
#pragma unroll
      for (int k = 0; k < WC / 4; ++k) {
        const float4 bb = b4[k];
        v[4 * k] += bb.x; v[4 * k + 1] += bb.y; v[4 * k + 2] += bb.z; v[4 * k + 3] += bb.w;
      }
      if (bias_smp && valid) {
#pragma unroll
        for (int j = 0; j < WC; ++j) { const int c = (n_off + n0 + j) % p.C_out; v[j] += __ldg(bias_smp + c); }
      }
    };

    // the whole column slice of this thread for one compile-time (GN, ACT, FILM) combination
    auto run = [&](auto gn_tag, auto act_tag, auto film_tag) {
      constexpr bool GN = decltype(gn_tag)::value;
      if constexpr (GN && N >= 32 && (Cfg::kCols / 8) > 32) {
        // wide layers (C_out = 512 / 1024: ChiUNet1d): a GroupNorm group is 64 / 128 columns -- too many to hold in registers,
        // so the group is read from TMEM twice: statistics first, then normalise + activation + store, 32 columns at a time
        constexpr int CPG = Cfg::kCols / 8;
        constexpr int GPT = NH / CPG;                 // whole groups per thread
        static_assert(NH % CPG == 0 && GPT >= 1, "a thread's column slice must hold whole GroupNorm groups");
        const float inv_cnt = 1.f / (float)(p.L * CPG);
#pragma unroll 1
        for (int g = 0; g < GPT; ++g) {
          float s1[1] = {0.f}, s2[1] = {0.f}, ga[1], gc[1];
#pragma unroll 1
          for (int ch = 0; ch < CPG / 32; ++ch) {
            const int n0 = col0 + g * CPG + ch * 32;
            float v[32];
            ptx::tmem_ld<32>(t_row + (uint32_t)n0, v);
            add_bias(std::integral_constant<int, 32>{}, v, n0);
#pragma unroll
            for (int j = 0; j < 32; ++j) { s1[0] += v[j]; s2[0] = fmaf(v[j], v[j], s2[0]); }
          }
          gn_coeffs<1>(s1, s2, p.L, p.log2L, lane, inv_cnt, p.gn_eps, ga, gc);
#pragma unroll 1
          for (int ch = 0; ch < CPG / 32; ++ch) {
            const int n0 = col0 + g * CPG + ch * 32;
            float v[32];
            ptx::tmem_ld<32>(t_row + (uint32_t)n0, v);
            add_bias(std::integral_constant<int, 32>{}, v, n0);
            const float4* ga4 = reinterpret_cast<const float4*>(&s_col[1][n_off + n0]);
            const float4* be4 = reinterpret_cast<const float4*>(&s_col[2][n_off + n0]);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const float4 gm = ga4[k], be = be4[k];
              v[4 * k + 0] = fmaf(fmaf(v[4 * k + 0], ga[0], gc[0]), gm.x, be.x);
              v[4 * k + 1] = fmaf(fmaf(v[4 * k + 1], ga[0], gc[0]), gm.y, be.y);
              v[4 * k + 2] = fmaf(fmaf(v[4 * k + 2], ga[0], gc[0]), gm.z, be.z);
              v[4 * k + 3] = fmaf(fmaf(v[4 * k + 3], ga[0], gc[0]), gm.w, be.w);
            }
            post16(act_tag, film_tag, v, std::integral_constant<int, 0>{}, n0);
            post16(act_tag, film_tag, v, std::integral_constant<int, 16>{}, n0 + 16);
          }
        }
      } else if constexpr (GN && N >= 32) {
        // GroupNorm (8 groups over the layer's kCols columns).  A chunk of WC = max(16, CPG) columns is read from TMEM
        // once and holds GPC = WC / CPG whole groups: per-thread sums over the group's columns, all-reduce over the L
        // lanes (= positions) of the trajectory, then y = ((v - mean) * rstd) * gamma + beta as two FMAs per element.
        constexpr int CPG = Cfg::kCols / 8;
        constexpr int WC = CPG > 16 ? CPG : 16;
        constexpr int GPC = WC / CPG;
        const float inv_cnt = 1.f / (float)(p.L * CPG);
#pragma unroll 1
        for (int ch = 0; ch < NH / WC; ++ch) {
          const int n0 = col0 + ch * WC;
          float v[WC];
          ptx::tmem_ld<WC>(t_row + (uint32_t)n0, v);
          add_bias(std::integral_constant<int, WC>{}, v, n0);
          float s1[GPC], s2[GPC], ga[GPC], gc[GPC];
#pragma unroll
          for (int g = 0; g < GPC; ++g) {
            s1[g] = 0.f; s2[g] = 0.f;
#pragma unroll
            for (int j = 0; j < CPG; ++j) { const float x = v[g * CPG + j]; s1[g] += x; s2[g] = fmaf(x, x, s2[g]); }
          }
          gn_coeffs<GPC>(s1, s2, p.L, p.log2L, lane, inv_cnt, p.gn_eps, ga, gc);
          const float4* ga4 = reinterpret_cast<const float4*>(&s_col[1][n_off + n0]);
          const float4* be4 = reinterpret_cast<const float4*>(&s_col[2][n_off + n0]);
#pragma unroll
          for (int k = 0; k < WC / 4; ++k) {
            const float4 gm = ga4[k], be = be4[k];
            const int g = (4 * k) / CPG;
            v[4 * k + 0] = fmaf(fmaf(v[4 * k + 0], ga[g], gc[g]), gm.x, be.x);
            v[4 * k + 1] = fmaf(fmaf(v[4 * k + 1], ga[g], gc[g]), gm.y, be.y);
            v[4 * k + 2] = fmaf(fmaf(v[4 * k + 2], ga[g], gc[g]), gm.z, be.z);
            v[4 * k + 3] = fmaf(fmaf(v[4 * k + 3], ga[g], gc[g]), gm.w, be.w);
          }
          post16(act_tag, film_tag, v, std::integral_constant<int, 0>{}, n0);
          if constexpr (WC == 32) post16(act_tag, film_tag, v, std::integral_constant<int, 16>{}, n0 + 16);
        }
      } else {
#pragma unroll 1
        for (int ch = 0; ch < NH / 16; ++ch) {
          float v[16];
          ptx::tmem_ld<16>(t_row + (uint32_t)(col0 + ch * 16), v);
          add_bias(std::integral_constant<int, 16>{}, v, col0 + ch * 16);
          post16(act_tag, film_tag, v, std::integral_constant<int, 0>{}, col0 + ch * 16);
        }
      }
    };

    if (active) {
      using T = std::true_type;
      using F = std::false_type;
      using A0 = std::integral_constant<int, CDS_ACT_NONE>;
      using A1 = std::integral_constant<int, CDS_ACT_MISH>;
      using AX = std::integral_constant<int, kActOther>;
      using F0 = std::integral_constant<int, 0>;
      using F1 = std::integral_constant<int, 1>;
      using F2 = std::integral_constant<int, 2>;
      if (has_gn) {
        if constexpr (Cfg::kGnOk) {
          if (p.act == CDS_ACT_MISH) {
            if (film == 0) run(T{}, A1{}, F0{});
            else if (film == 1) run(T{}, A1{}, F1{});
            else run(T{}, A1{}, F2{});
          } else {
            run(T{}, AX{}, F2{});
          }
        }
      } else {
        if (p.act == CDS_ACT_NONE && film == 0) run(F{}, A0{}, F0{});
        else run(F{}, AX{}, F2{});
      }
    }
    // hand the accumulator buffer back to the MMA warp (one arrival per epilogue warp)
    ptx::tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&tmem_empty_bar[buf]);
    if (threadIdx.x == 0 && it < 14) CDS_TRACE(11 + 4 * it, clock64());
    }   // tile loop
    if (threadIdx.x == 0) CDS_TRACE(5, (long long)it);
  }

  // bulk stores issued by the epilogue warps' lane 0 must be complete (shared memory read AND global writes performed) before
  // the CTA retires
  if (warp < kTcEpiThreads / 32 && lane == 0) ptx::bulk_wait_group<0>();
  __syncthreads();
  if (cs > 1) ptx::cluster_sync();                    // no CTA retires while a peer may still multicast into it / signal its barriers
  if (warp == 9) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
  if (threadIdx.x == 0) { CDS_TRACE(3, clock64()); CDS_TRACE(4, gtimer()); }
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(ptr);
  }
  return fn;
}

// bf16 (tf32 = false) or fp32 (tf32 = true) tensor, dims innermost-first; strides in elements for dims 1.. (dim 0 is
// contiguous); kc = row bytes / 2 of the box (64: SWIZZLE_128B, 32: SWIZZLE_64B), box[0] = kc (bf16) or kc / 2 (fp32) elements
inline bool encode_act_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_el,
                           const uint32_t* box, int kc, bool tf32, const uint32_t* elem_strides = nullptr) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return false;
  cuuint64_t gdim[3], gstr[2];
  cuuint32_t bx[3], es[3];
  const int eb = tf32 ? 4 : 2;
  for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; es[i] = elem_strides ? elem_strides[i] : 1; }
  for (int i = 1; i < rank; ++i) gstr[i - 1] = strides_el[i - 1] * eb;
  CUtensorMapSwizzle sw = kc == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = enc(m, tf32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank,
                   const_cast<void*>(base), gdim, gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

inline int ilog2(int v) { int r = 0; while ((1 << r) < v) ++r; return r; }

inline bool conv_is_tf32(const cds_conv_op& c) { return c.math == CDS_MATH_TF32_TC; }
// operand row width in bf16-equivalents (row bytes / 2): 64 (128-byte rows, SWIZZLE_128B) when every K extent fills whole
// 128-byte rows (64 bf16 / 32 fp32 channels), else 32 (64-byte rows, SWIZZLE_64B: 32 bf16 / 16 fp32 channels)
inline int conv_tc_pick_kc(const cds_conv_op& c) {
  const int full = conv_is_tf32(c) ? 32 : 64;
  bool wide = (c.C_in % full == 0) && (!c.res_w || c.res_C % full == 0);
  return wide ? 64 : 32;
}

// GEMM width of the op: C_out*phases, or 16 for a narrow (C_out <= 16) 1x1 head whose missing weight rows the TMA
// unit zero-fills (out-of-bound rows of the weight tensor); 0 = not a width the kernel is instantiated for
// column-tile width for the runtime-tiled (un-normalised) layers of total width n (a multiple of 64): the widest instantiated
// tile that divides it -- wide tiles re-load the activation tile less often (DiT1d: 1280 = 5 x 256, 960 = 5 x 192, 320 = 2 x 160)
// (the 160 / 192-wide tiles are instantiated for 128-byte operand rows only: kc == 64)
inline int conv_tc_runtime_tile(int n, int kc) {
  if (n % 256 == 0) return 256;
  if (kc == 64 && n % 192 == 0) return 192;
  if (kc == 64 && n % 160 == 0) return 160;
  return n % 128 == 0 ? 128 : 64;
}
inline int conv_tc_width(const cds_conv_op& c) {
  int n = c.C_out * c.phases;
  if (n == 32 || n == 64 || n == 128 || n == 256) return (c.phases == 1 || c.C_out % 16 == 0) ? n : 0;
  if ((n == 512 || n == 1024) && c.phases == 1) return n;      // wide layers: 2 / 4 CTAs of 256 columns (2-4 whole GroupNorm groups each)
  // un-normalised layers of any width that is a multiple of 64 (DiT1d's 320 / 960 / 1280-wide Linear layers): runtime column tiles
  if (n > 64 && n % 64 == 0 && c.groups == 0) {
    const int tn = conv_tc_runtime_tile(n, conv_tc_pick_kc(c));           // a column tile must not straddle the two phases
    if (c.phases == 1 || c.C_out % tn == 0) return n;
  }
  // narrow output heads (C_out <= 32, e.g. 14 / 29 state dims): N = 16 / 32 with the missing weight rows zero-filled by the TMA unit
  if (n <= 32 && n != 32 && c.phases == 1 && c.taps == 1 && c.groups == 0 && !c.res_w && !c.res) return n <= 16 ? 16 : 32;
  return 0;
}

// can the tensor-core kernel serve this op?  (otherwise the fp32 CUDA-core kernel runs it, any dtype)
inline bool conv_tc_eligible(const cds_conv_op& c) {
  if (c.math != CDS_MATH_BF16_TC && c.math != CDS_MATH_TF32_TC) return false;
  const bool tf32 = conv_is_tf32(c);
  // operand tensors (in, res_in) must have the mode's storage type: bf16, or fp32 (CDS_F32 / CDS_TF32 read alike)
  auto operand_ok = [tf32](int dt) { return tf32 ? (dt == CDS_F32 || dt == CDS_TF32) : (dt == CDS_BF16); };
  const int vec_el = tf32 ? 4 : 8;                    // elements per 16 bytes
  const int kmin = tf32 ? 16 : 32;                    // channels in a 64-byte operand row
  if (!operand_ok(c.in_dtype)) return false;
  if (c.stride != 1 && c.stride != 2) return false;
  if (c.phases != 1 && c.phases != 2) return false;
  int L = c.L_out;                                   // tile rows = 128/L trajectories x L output positions
  if (L > 32 || (L & (L - 1)) != 0) return false;
  if (c.stride == 1 ? (c.L_in != L) : (c.L_in != 2 * L || c.phases != 1 || c.res_w || c.res)) return false;
  if (conv_tc_width(c) == 0) return false;
  if (conv_tc_width(c) > 256 && c.groups != 0 && conv_tc_pick_kc(c) != 64) return false;   // wide GN variants: KC = 64 only
  if (c.sample_row_div > 1 && c.L_out != 1) return false;
  if (c.C_in % kmin != 0) return false;
  if (c.groups != 0 && (c.groups != 8 || c.phases != 1 || c.C_out < 32)) return false;
  if (c.phases == 2 && (c.res || c.res_w)) return false;
  int T = 128 / L;
  if (c.in_batch_mod > 0 && c.in_batch_mod % T != 0) return false;
  if (c.res_batch_mod > 0 && c.res_w && c.res_batch_mod % T != 0) return false;   // (the identity residual is read row by row)
  if (c.res_w && (!operand_ok(c.res_in_dtype) || c.res_C % kmin != 0)) return false;
  if ((c.in_lstride % vec_el) || (c.in_bstride % vec_el) || ((uintptr_t)c.in % 16)) return false;
  if (c.res_w && ((c.res_in_lstride % vec_el) || (c.res_in_bstride % vec_el) || ((uintptr_t)c.res_in % 16))) return false;
  if (c.C_out % 16 == 0) {                           // vector stores
    if (c.out_dtype == 1 ? ((c.out_lstride % 8) || ((uintptr_t)c.out % 16)) : ((c.out_lstride % 4) || ((uintptr_t)c.out % 16)))
      return false;
  }
  if (c.res && (c.res_dtype == 1 ? ((c.res_lstride % 8) || ((uintptr_t)c.res % 16)) : ((c.res_lstride % 4) || ((uintptr_t)c.res % 16))))
    return false;
  return true;
}

struct ConvTcLaunch {
  ConvTcParams prm;
  bool tf32 = false;              // fp32 operands read as TF32 (CDS_MATH_TF32_TC)
  int kc = 0, n = 0, split = 1;   // n = CTA tile width, split*n = layer width
  int max_ctas_per_sm = 0;        // > 0: use at most this many CTAs per SM (plans with parallel branches share the SMs)
  bool has_res = false;
  dim3 grid;
};

// Share a layer's columns between two CTAs?  Yes for the wide layers (C_out >= 128: halves the per-CTA epilogue and main
// loop and lets two CTAs share an SM) and for C_out = 64 when there are too few row tiles to fill the machine.
inline int conv_tc_pick_split(const cds_conv_op& c, int n_total, int m_tiles) {
  if (n_total > 256) return n_total / 256;
  if (c.phases != 1 || n_total < 64) return 1;
  if (const char* ns = getenv("CDS_TC_NOSPLIT")) { if (ns[0] == '1') return 1; if (ns[0] == '2' && n_total == 128) return 1; }   // experiment
  if (n_total >= 128) return 2;
  // TF32 programs: two 32-wide CTAs fetch the (fp32) activation tile twice, and the kernels are bound by the L2 -> SM feed of
  // their operand tiles (DESIGN.md section 5), so the 64-wide layers stay whole even when that leaves fewer tiles than CTA slots
  // (cfg2, TF32: 597 vs 608 us per iteration)
  if (conv_is_tf32(c)) return 1;
  const char* e = getenv("CDS_TC_SPLIT64");
  if (e && e[0] == '1') return 2;                    // experiment: C_out = 64 always as two N = 32 CTAs (3 CTAs/SM residency)
  return m_tiles < 296 ? 2 : 1;
}

inline bool conv_tc_prepare(const cds_conv_op& c, ConvTcLaunch* out) {
  ConvTcLaunch& L = *out;
  memset(&L.prm, 0, sizeof(L.prm));
  const int kc = conv_tc_pick_kc(c);
  const bool tf32 = conv_is_tf32(c);
  const int ke = tf32 ? kc / 2 : kc;                   // channels per chunk
  L.tf32 = tf32;
  ConvTcParams& p = L.prm;
  const int Lp = c.L_out, T = 128 / Lp;
  const int64_t rows = (int64_t)c.batch * Lp;
  const int m_tiles = (int)((rows + 127) / 128);
  const int n_total = conv_tc_width(c);
  L.kc = kc; L.has_res = c.res_w != nullptr;
  int col_tiles = 1;                                  // runtime column tiles (SPLIT == 1 kernels)
  const bool fixed = n_total == 16 || n_total == 32 || n_total == 64 || n_total == 128 || n_total == 256 ||
                     ((n_total == 512 || n_total == 1024) && c.groups != 0);
  if (fixed) {
    L.split = conv_tc_pick_split(c, n_total, m_tiles);
    L.n = n_total / L.split;
  } else {
    L.split = 1;
    L.n = conv_tc_runtime_tile(n_total, kc);
    col_tiles = n_total / L.n;
  }
  const uint64_t in_b = c.in_batch_mod > 0 ? (uint64_t)c.in_batch_mod : (uint64_t)c.batch;
  {
    uint64_t dims[3] = {(uint64_t)c.C_in, (uint64_t)c.L_in, in_b};
    uint64_t str[2] = {(uint64_t)c.in_lstride, (uint64_t)c.in_bstride};
    // stride-2 conv: the box walks the position axis with element stride 2 (box extent = 2*L traversed -> L loaded)
    uint32_t box[3] = {(uint32_t)ke, (uint32_t)(Lp * c.stride), (uint32_t)T};
    uint32_t es[3] = {1u, (uint32_t)c.stride, 1u};
    if (!encode_act_map(&p.tm_a, c.in, 3, dims, str, box, kc, tf32, es)) return false;
  }
  {
    // weight rows beyond taps*C_out*phases (narrow heads padded to N=16) are zero-filled by the TMA unit
    uint64_t dims[2] = {(uint64_t)c.C_in, (uint64_t)c.taps * c.C_out * c.phases};
    uint64_t str[1] = {(uint64_t)c.C_in};
    uint32_t box[2] = {(uint32_t)ke, (uint32_t)L.n};
    if (!encode_act_map(&p.tm_b, c.w, 2, dims, str, box, kc, tf32)) return false;
  }
  // Opt-in (CDS_MULTICAST=1).  Measured on B200 (cfg2, batch 4096): 636 vs 615 us per iteration in TF32, 474 vs 452 in bf16 --
  // what binds the main loop is the bytes INGESTED into each SM's shared memory (TMA fill + MMA operand reads, ~128 B/clk/SM),
  // which multicast does not reduce, while the lock-step of the cluster costs a little.
  { const char* mc = getenv("CDS_MULTICAST"); p.cluster = (L.split > 1 && T % L.split == 0 && mc && mc[0] == '1') ? L.split : 1; }
  if (p.cluster > 1) {      // the activation tensor again, with the box of ONE cluster CTA's share of the tile's trajectories
    uint64_t dims[3] = {(uint64_t)c.C_in, (uint64_t)c.L_in, in_b};
    uint64_t str[2] = {(uint64_t)c.in_lstride, (uint64_t)c.in_bstride};
    uint32_t box[3] = {(uint32_t)ke, (uint32_t)(Lp * c.stride), (uint32_t)(T / L.split)};
    uint32_t es[3] = {1u, (uint32_t)c.stride, 1u};
    if (!encode_act_map(&p.tm_a_mc, c.in, 3, dims, str, box, kc, tf32, es)) return false;
  }
  if (L.has_res) {
    const uint64_t r_b = c.res_batch_mod > 0 ? (uint64_t)c.res_batch_mod : (uint64_t)c.batch;
    uint64_t dims[3] = {(uint64_t)c.res_C, (uint64_t)Lp, r_b};
    uint64_t str[2] = {(uint64_t)c.res_in_lstride, (uint64_t)c.res_in_bstride};
    uint32_t box[3] = {(uint32_t)ke, (uint32_t)Lp, (uint32_t)T};
    if (!encode_act_map(&p.tm_a2, c.res_in, 3, dims, str, box, kc, tf32)) return false;
    if (p.cluster > 1) {
      uint32_t boxp[3] = {(uint32_t)ke, (uint32_t)Lp, (uint32_t)(T / L.split)};
      if (!encode_act_map(&p.tm_a2_mc, c.res_in, 3, dims, str, boxp, kc, tf32)) return false;
    }
    uint64_t d2[2] = {(uint64_t)c.res_C, (uint64_t)c.C_out};
    uint64_t s2[1] = {(uint64_t)c.res_C};
    uint32_t b2[2] = {(uint32_t)ke, (uint32_t)L.n};
    if (!encode_act_map(&p.tm_b2, c.res_w, 2, d2, s2, b2, kc, tf32)) return false;
  }
  {
    // output as a TMA-store target (the fast epilogue lanes stage 32 rows x 16 columns per warp and bulk-store them): needs whole
    // 16-column groups, 16-byte aligned rows, one phase, at most 32 positions per trajectory
    const int oes = c.out_dtype == CDS_BF16 ? 2 : 4;
    const bool ok = (c.phases == 1 || c.phases == 2) && c.C_out % 16 == 0 && Lp <= 32 && ((uintptr_t)c.out % 16) == 0 &&
                    ((int64_t)c.out_lstride * oes) % 16 == 0 && ((int64_t)c.out_bstride * oes) % 16 == 0 && !getenv("CDS_NO_TMA_STORE");
    p.out_tma = 0;
    if (ok) {
      PFN_encodeTiled enc = get_encode_tiled();
      const CUtensorMapDataType dt = oes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
      const CUtensorMapSwizzle sw = oes == 2 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_64B;
      if (c.phases == 1) {
        cuuint64_t gdim[3] = {(cuuint64_t)c.C_out, (cuuint64_t)Lp, (cuuint64_t)c.batch};
        cuuint64_t gstr[2] = {(cuuint64_t)c.out_lstride * oes, (cuuint64_t)c.out_bstride * oes};
        cuuint32_t bx[3] = {16u, (cuuint32_t)Lp, (cuuint32_t)(32 / Lp)};
        cuuint32_t es[3] = {1u, 1u, 1u};
        if (enc && enc(&p.tm_out, dt, 3, c.out, gdim, gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                       CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
          p.out_tma = 1;
      } else {
        // two-phase transposed conv: tile row (trajectory, l) writes output position 2l + phase -> the output seen as
        // {C, phase, L, batch} with strides {lstride, 2 lstride, bstride}; a store box covers ONE phase of its 32 rows
        cuuint64_t gdim[4] = {(cuuint64_t)c.C_out, 2u, (cuuint64_t)Lp, (cuuint64_t)c.batch};
        cuuint64_t gstr[3] = {(cuuint64_t)c.out_lstride * oes, (cuuint64_t)c.out_lstride * 2 * oes, (cuuint64_t)c.out_bstride * oes};
        cuuint32_t bx[4] = {16u, 1u, (cuuint32_t)Lp, (cuuint32_t)(32 / Lp)};
        cuuint32_t es[4] = {1u, 1u, 1u, 1u};
        if (enc && enc(&p.tm_out, dt, 4, c.out, gdim, gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                       CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
          p.out_tma = 2;
      }
    }
  }
  p.res_tma = 0;
  if (c.res && !c.res_w && c.res_batch_mod == 0 && c.phases == 1 && c.C_out % 16 == 0 && Lp <= 32 && L.n <= 64 &&
      c.res_dtype == (tf32 ? c.res_dtype : CDS_BF16) && (tf32 ? c.res_dtype != CDS_BF16 : true) && !getenv("CDS_NO_TMA_RES")) {
    const int res_es = tf32 ? 4 : 2;
    if (((uintptr_t)c.res % 16) == 0 && ((int64_t)c.res_lstride * res_es) % 16 == 0 && ((int64_t)c.res_bstride * res_es) % 16 == 0) {
      PFN_encodeTiled enc = get_encode_tiled();
      cuuint64_t gdim[3] = {(cuuint64_t)c.C_out, (cuuint64_t)Lp, (cuuint64_t)c.batch};
      cuuint64_t gstr[2] = {(cuuint64_t)c.res_lstride * res_es, (cuuint64_t)c.res_bstride * res_es};
      cuuint32_t bx[3] = {16u, (cuuint32_t)Lp, (cuuint32_t)(32 / Lp)};
      cuuint32_t es[3] = {1u, 1u, 1u};
      if (enc && enc(&p.tm_res, tf32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(c.res), gdim,
                     gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, tf32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B,
                     CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
        p.res_tma = 1;
    }
  }
  p.batch = c.batch; p.L = Lp; p.log2L = ilog2(Lp); p.C_out = c.C_out; p.taps = c.taps; p.pad = c.pad;
  p.phases = c.phases;
  p.kchunks = c.C_in / ke; p.kchunks2 = L.has_res ? c.res_C / ke : 0;
  p.in_batch_mod = c.in_batch_mod;
  p.bias = c.bias; p.scale = c.scale; p.shift = c.shift;
  p.groups = c.groups; p.gn_gamma = c.gn_gamma; p.gn_beta = c.gn_beta; p.gn_eps = c.gn_eps; p.act = c.act;
  p.res = c.res; p.res_bstride = c.res_bstride; p.res_lstride = c.res_lstride; p.res_batch_mod = c.res_batch_mod;
  p.res_dtype = c.res_dtype; p.res_bias = c.res_bias;
  p.out = c.out; p.out_bstride = c.out_bstride; p.out_lstride = c.out_lstride; p.out_dtype = c.out_dtype;
  p.n_col_tiles = col_tiles;
  p.sample_div = c.sample_row_div > 1 ? c.sample_row_div : 1;
  p.num_tiles = m_tiles * (L.split > 1 ? L.split : col_tiles);
  L.grid = dim3((unsigned)p.num_tiles);      // clipped to the resident-CTA capacity at launch (persistent CTAs)
  return true;
}

// debug: returns the trace buffer if THIS tensor-core launch is the one selected by cds_debug_trace (cds_api.cu), else NULL
long long* conv_tc_trace_hook(int grid);

// Launch wrapper of one instantiation.  The instantiations are compiled in conv_tc_inst.cu (several translation units, built
// in parallel); every other translation unit only sees the extern declarations below.
template <int KC, int N, bool HAS_RES, int SPLIT, bool TF32>
cudaError_t conv_tc_launch_t(const ConvTcLaunch& L, const int* iter_ptr, cudaStream_t st) {
  using Cfg = ConvTcCfg<KC, N, HAS_RES, SPLIT>;
  static bool attr = false;
  static int resident = 0;                   // CTAs of this instantiation that fit on the device at once
  static int sm_count = 0;
  static bool pdl = true;                    // chain with programmatic dependent launch (CDS_PDL=0: plain stream order)
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel<KC, N, HAS_RES, SPLIT, TF32>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Cfg::kSmemBytes);
    if (e != cudaSuccess) return e;
    // several CTAs per SM for the narrow tiles: ask for the maximum shared-memory carve-out
    e = cudaFuncSetAttribute(conv_tc_kernel<KC, N, HAS_RES, SPLIT, TF32>, cudaFuncAttributePreferredSharedMemoryCarveout,
                             cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // residency we design for: launch-bounds blocks, TMEM (kTmemCols of 512 columns per SM), 227 KB shared memory
    int want = Cfg::kMinBlocks;
    int by_tmem = 512 / (int)Cfg::kTmemCols;
    // static shared memory: 16 KB store staging + 24 B/column of constants + barriers (+ 16 KB residual staging), 1 KB reserved
    const int static_smem = 16 * 1024 + 24 * Cfg::kCols + 1024 + (Cfg::kResStage ? 16 * 1024 : 0) + 1024;
    int by_smem = (227 * 1024) / (Cfg::kSmemBytes + static_smem);
    if (want > by_tmem) want = by_tmem;
    if (want > by_smem) want = by_smem;
    if (const char* cap = getenv("CDS_TC_MAXCTAS")) { int c = atoi(cap); if (c >= 1 && c < want) want = c; }
    if (want < 1) want = 1;
    if (getenv("CDS_DEBUG"))
      fprintf(stderr, "[cds] conv_tc<%d,%d,%d,%d,%s>: designed %d CTA/SM (tmem %d, smem %d), smem %d B, %d stages\n", KC, N,
              (int)HAS_RES, SPLIT, TF32 ? "tf32" : "bf16", want, by_tmem, by_smem, Cfg::kSmemBytes, Cfg::kStages);
    resident = want * sms;
    sm_count = sms;
    const char* pdl_env = getenv("CDS_PDL");
    pdl = !(pdl_env && pdl_env[0] == '0');
    attr = true;
  }
  unsigned cap = (unsigned)resident;
  if (L.max_ctas_per_sm > 0 && (unsigned)(L.max_ctas_per_sm * sm_count) < cap) cap = (unsigned)(L.max_ctas_per_sm * sm_count);
  dim3 grid(L.grid.x < cap ? L.grid.x : cap);
  const unsigned cl = L.prm.cluster > 1 ? (unsigned)L.prm.cluster : 1u;
  if (cl > 1) grid.x -= grid.x % cl;                 // whole clusters: the CTAs of a cluster walk the same row tiles in lockstep
  ConvTcParams prm = L.prm;
  prm.trace = conv_tc_trace_hook((int)grid.x);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = dim3(kTcThreads); cfg.dynamicSmemBytes = Cfg::kSmemBytes; cfg.stream = st;
  cudaLaunchAttribute at[2];
  int na = 0;
  if (pdl) { at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[na].val.programmaticStreamSerializationAllowed = 1; ++na; }
  if (cl > 1) {
    at[na].id = cudaLaunchAttributeClusterDimension;
    at[na].val.clusterDim.x = cl; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
    ++na;
  }
  cfg.attrs = at; cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, conv_tc_kernel<KC, N, HAS_RES, SPLIT, TF32>, prm, iter_ptr);
}
// touch the kernel once (module load) so that nothing lazy happens inside a stream capture
template <int KC, int N, bool HAS_RES, int SPLIT, bool TF32>
cudaError_t conv_tc_preload_t() {
  cudaFuncAttributes a;
  return cudaFuncGetAttributes(&a, conv_tc_kernel<KC, N, HAS_RES, SPLIT, TF32>);
}

// every (KC, N, SPLIT) the dispatcher can pick (each with and without the shortcut accumulator); X(kc, n, split)
#define CDS_TC_VARIANTS(X)                                                                              \
  X(64, 16, 1) X(64, 32, 1) X(64, 64, 1) X(64, 128, 1) X(64, 256, 1) X(64, 32, 2) X(64, 64, 2) X(64, 128, 2) \
  X(64, 256, 2) X(64, 256, 4) X(64, 160, 1) X(64, 192, 1)                                                \
  X(32, 16, 1) X(32, 32, 1) X(32, 64, 1) X(32, 128, 1) X(32, 256, 1) X(32, 32, 2) X(32, 64, 2) X(32, 128, 2)

#ifndef CDS_TC_INSTANTIATE
#define CDS_TC_EXTERN2(KC_, N_, S_, T_)                                                                                 \
  extern template cudaError_t conv_tc_launch_t<KC_, N_, false, S_, T_>(const ConvTcLaunch&, const int*, cudaStream_t);  \
  extern template cudaError_t conv_tc_launch_t<KC_, N_, true, S_, T_>(const ConvTcLaunch&, const int*, cudaStream_t);   \
  extern template cudaError_t conv_tc_preload_t<KC_, N_, false, S_, T_>();                                              \
  extern template cudaError_t conv_tc_preload_t<KC_, N_, true, S_, T_>();
#define CDS_TC_EXTERN(KC_, N_, S_) CDS_TC_EXTERN2(KC_, N_, S_, false) CDS_TC_EXTERN2(KC_, N_, S_, true)
CDS_TC_VARIANTS(CDS_TC_EXTERN)
#undef CDS_TC_EXTERN
#undef CDS_TC_EXTERN2

inline cudaError_t conv_tc_launch(const ConvTcLaunch& L, const int* iter_ptr, cudaStream_t st) {
#define CDS_TC_CASE(KC_, N_, S_)                                                                                         \
  if (L.kc == KC_ && L.n == N_ && L.split == S_) {                                                                       \
    if (L.tf32) return L.has_res ? conv_tc_launch_t<KC_, N_, true, S_, true>(L, iter_ptr, st)                            \
                                 : conv_tc_launch_t<KC_, N_, false, S_, true>(L, iter_ptr, st);                          \
    return L.has_res ? conv_tc_launch_t<KC_, N_, true, S_, false>(L, iter_ptr, st)                                       \
                     : conv_tc_launch_t<KC_, N_, false, S_, false>(L, iter_ptr, st);                                     \
  }
  CDS_TC_VARIANTS(CDS_TC_CASE)
#undef CDS_TC_CASE
  return cudaErrorInvalidValue;
}

inline cudaError_t conv_tc_preload_all() {
  cudaError_t e;
#define CDS_TC_PRE(KC_, N_, S_)                                                              \
  if ((e = conv_tc_preload_t<KC_, N_, false, S_, false>()) != cudaSuccess) return e;         \
  if ((e = conv_tc_preload_t<KC_, N_, true, S_, false>()) != cudaSuccess) return e;          \
  if ((e = conv_tc_preload_t<KC_, N_, false, S_, true>()) != cudaSuccess) return e;          \
  if ((e = conv_tc_preload_t<KC_, N_, true, S_, true>()) != cudaSuccess) return e;
  CDS_TC_VARIANTS(CDS_TC_PRE)
#undef CDS_TC_PRE
  return cudaSuccess;
}
#endif  // !CDS_TC_INSTANTIATE

}  // namespace cds
