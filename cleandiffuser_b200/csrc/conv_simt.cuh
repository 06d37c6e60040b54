// CDS_OP_CONV, fp32 CUDA-core path: implicit-GEMM 1-D convolution / linear layer with the whole
// post-processing of a UNet conv block fused behind it.
//
//   rows    M = batch * L_out        (one row per output position of one trajectory)
//   columns N = C_out * phases
//   depth   K = taps * C_in          (im2col is formed on the fly from the channels-last activation)
//
// One CTA owns a 128 x BN tile.  128 rows are whole trajectories (L_out | 128) and BN is a multiple of
// the GroupNorm group width, so every (trajectory, group) whose statistics are needed lives inside ONE
// tile: the accumulators go to shared memory once, a warp per (trajectory, group) reduces mean / variance
// with shuffles, and a coalesced pass applies GN-affine, Mish, FiLM and the residual and stores -- the
// conv output never makes an HBM round trip before its normalisation.  An optional second, short GEMM
// (the 1x1 shortcut conv of a ResidualBlock) is accumulated on top of the finished tile.
//
// Algorithmic HBM bytes per launch: 4*(batch*L_in*C_in + batch*L_out*C_out*phases) (+ shortcut input, +weights
// once per CTA column through L2).  The tcgen05 path (conv_tc.cuh) replaces the main loop; the epilogue is shared.
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace cds {

constexpr int kBM = 128;      // rows per CTA tile
constexpr int kBK = 16;       // depth per smem stage
constexpr int kThreads = 256; // 16 x 16 thread grid, each thread an 8 x (BN/16) register tile
constexpr int kAPad = 4;

__device__ __forceinline__ float ld_act(const void* base, int64_t idx, int dtype) {
  return dtype == CDS_BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[idx])
                           : __ldg(reinterpret_cast<const float*>(base) + idx);
}
__device__ __forceinline__ void st_act(void* base, int64_t idx, int dtype, float v) {
  if (dtype == CDS_BF16) reinterpret_cast<__nv_bfloat16*>(base)[idx] = __float2bfloat16_rn(v);
  else if (dtype == CDS_TF32) reinterpret_cast<float*>(base)[idx] = round_tf32(v);
  else reinterpret_cast<float*>(base)[idx] = v;
}

struct ConvSrc {              // one im2col source (main conv, or the 1x1 shortcut)
  const void* in; int dtype; int64_t bstride; int lstride; int bmod;
  int C, taps, stride, pad, L_in;
  const float* w;             // [taps*C][N]
};

template <int BN>
struct ConvSmem {
  static constexpr int kTN = BN / 16;
  static constexpr int kAs = kBK * (kBM + kAPad);
  static constexpr int kBs = kBK * BN;
  static constexpr int kCs = kBM * (BN + 1);
  static constexpr int kStats = kBM * 8 * 2;   // <= 128 trajectories x <= 8 groups x (mean, rstd)
  static constexpr size_t bytes = sizeof(float) * (kAs + kBs + kCs + kStats);
};

// acc += A(rows, K) * W(K, cols) for this CTA's tile; A gathered from `s` (zero padded), register-prefetched.
template <int BN>
__device__ __forceinline__ void gemm_mainloop(const ConvSrc& s, float (&acc)[8][BN / 16], float* As, float* Bs,
                                              const int (&row_b)[8], const int (&row_l)[8], int n0, int N_total) {
  constexpr int TN = BN / 16;
  constexpr int kBLoads = (kBK * BN) / kThreads;   // B elements each thread stages per chunk
  const int t = threadIdx.x;
  const int tx = t & 15, ty = t >> 4;
  const int a_kk = t & 15;          // this thread stages depth index a_kk of rows (t>>4) + 16*j
  const int K_total = s.taps * s.C;

  // per-row gather bases (row_b < 0 marks a row outside the problem)
  int64_t a_base[8]; int a_pos0[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    int b = row_b[j];
    if (b >= 0) {
      int bb = s.bmod > 0 ? b % s.bmod : b;
      a_pos0[j] = row_l[j] * s.stride - s.pad;
      a_base[j] = (int64_t)bb * s.bstride;
    } else { a_pos0[j] = -(1 << 28); a_base[j] = 0; }
  }

  float a_reg[8], b_reg[kBLoads];
  auto fetch = [&](int k0) {
    int kg = k0 + a_kk;
    bool kv = kg < K_total;
    int tap = kv ? kg / s.C : 0;
    int ci = kg - tap * s.C;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int pos = a_pos0[j] + tap;
      bool ok = kv && pos >= 0 && pos < s.L_in;
      a_reg[j] = ok ? ld_act(s.in, a_base[j] + (int64_t)pos * s.lstride + ci, s.dtype) : 0.f;
    }
#pragma unroll
    for (int j = 0; j < kBLoads; ++j) {
      int idx = t + j * kThreads;
      int kk = idx / BN, n = idx - kk * BN;
      bool ok = (k0 + kk) < K_total && (n0 + n) < N_total;
      b_reg[j] = ok ? __ldg(s.w + (int64_t)(k0 + kk) * N_total + n0 + n) : 0.f;
    }
  };
  auto stage = [&]() {
#pragma unroll
    for (int j = 0; j < 8; ++j) As[a_kk * (kBM + kAPad) + (t >> 4) + 16 * j] = a_reg[j];
#pragma unroll
    for (int j = 0; j < kBLoads; ++j) Bs[t + j * kThreads] = b_reg[j];
  };

  fetch(0);
  stage();
  __syncthreads();
  for (int k0 = 0; k0 < K_total; k0 += kBK) {
    bool more = k0 + kBK < K_total;
    if (more) fetch(k0 + kBK);
#pragma unroll
    for (int kk = 0; kk < kBK; ++kk) {
      float a[8], b[TN];
      const float4* ap = reinterpret_cast<const float4*>(As + kk * (kBM + kAPad) + ty * 8);
      float4 a0 = ap[0], a1 = ap[1];
      a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w; a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
#pragma unroll
      for (int j = 0; j < TN; ++j) b[j] = Bs[kk * BN + tx * TN + j];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
    if (more) { stage(); __syncthreads(); }
  }
}

template <int BN>
__global__ void __launch_bounds__(kThreads) conv_gemm_f32_kernel(const cds_conv_op p, const int* __restrict__ iter_ptr) {
  constexpr int TN = BN / 16;
  extern __shared__ __align__(16) float smem[];
  float* As = smem;
  float* Bs = As + ConvSmem<BN>::kAs;
  float* Cs = Bs + ConvSmem<BN>::kBs;
  float* stats = Cs + ConvSmem<BN>::kCs;

  const int iter = iter_ptr ? *iter_ptr : 0;
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int rows = p.batch * p.L_out;
  const int N_total = p.C_out * p.phases;
  const int row0 = blockIdx.x * kBM;
  const int n0 = blockIdx.y * BN;

  // rows this thread STAGES for the gather: (t>>4) + 16*j
  int st_b[8], st_l[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    int r = row0 + (t >> 4) + 16 * j;
    if (r < rows) { st_b[j] = r / p.L_out; st_l[j] = r - st_b[j] * p.L_out; } else { st_b[j] = -1; st_l[j] = 0; }
  }

  float acc[8][TN];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  ConvSrc main_src{p.in, p.in_dtype, p.in_bstride, p.in_lstride, p.in_batch_mod, p.C_in, p.taps, p.stride, p.pad, p.L_in,
                   reinterpret_cast<const float*>(p.w)};
  gemm_mainloop<BN>(main_src, acc, As, Bs, st_b, st_l, n0, N_total);

  // ---- accumulators (+bias) -> shared tile -------------------------------------------------------
  const VecRef bias = resolve(p.bias, iter);
  // GroupNorm layers: the step bias minus its group mean (group_mean, common.cuh) -- the normalised output is the same, and the
  // fp32 mean of the statistics pass no longer carries the rounding of a large common offset
  float bias_shift[TN];
#pragma unroll
  for (int j = 0; j < TN; ++j) {
    const int ng = n0 + tx * TN + j;
    const int gcpg = p.groups > 0 ? p.C_out / p.groups : 0;
    bias_shift[j] = (gcpg && bias.step && ng < N_total) ? group_mean(bias.step, ng - ng % gcpg, gcpg) : 0.f;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int m = ty * 8 + i;
    int r = row0 + m;
    int b = r < rows ? r / p.L_out : 0;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      int n = tx * TN + j;
      int ng = n0 + n;
      float v = acc[i][j];
      if (r < rows && ng < N_total && bias.present()) {
        const int c = ng % p.C_out;
        if (bias.step) v += __ldg(bias.step + c) - bias_shift[j];
        if (bias.sample) v += __ldg(bias.sample + (int64_t)b * bias.sample_stride + c);
      }
      Cs[m * (BN + 1) + n] = v;
    }
  }
  __syncthreads();

  // ---- GroupNorm statistics: one warp per (trajectory, group) of the tile ---------------------------
  const int cpg = p.groups > 0 ? p.C_out / p.groups : 0;
  const int g_tile = p.groups > 0 ? min(BN, N_total - n0) / cpg : 0;
  if (p.groups > 0) {
    const int traj_tile = kBM / p.L_out;
    const int warp = t >> 5, lane = t & 31;
    const int cnt = p.L_out * cpg;
    for (int pair = warp; pair < traj_tile * g_tile; pair += kThreads / 32) {
      int tj = pair / g_tile, g = pair - tj * g_tile;
      const float* base = Cs + (tj * p.L_out) * (BN + 1) + g * cpg;
      float s = 0.f;
      for (int e = lane; e < cnt; e += 32) { int l = e / cpg, c = e - l * cpg; s += base[l * (BN + 1) + c]; }
      float mean = warp_sum(s) / (float)cnt;
      float q = 0.f;
      for (int e = lane; e < cnt; e += 32) {
        int l = e / cpg, c = e - l * cpg;
        float d = base[l * (BN + 1) + c] - mean;
        q = fmaf(d, d, q);
      }
      float var = warp_sum(q) / (float)cnt;
      if (lane == 0) { stats[pair * 2] = mean; stats[pair * 2 + 1] = rsqrtf(var + p.gn_eps); }
    }
    __syncthreads();
  }

  // ---- coalesced post-processing pass ---------------------------------------------------------------
  const VecRef scale = resolve(p.scale, iter), shift = resolve(p.shift, iter);
  const bool second_gemm = p.res_w != nullptr;
  for (int idx = t; idx < kBM * BN; idx += kThreads) {
    int m = idx / BN, n = idx - m * BN;
    int r = row0 + m, ng = n0 + n;
    if (r >= rows || ng >= N_total) continue;
    int b = r / p.L_out, l = r - b * p.L_out;
    int phase = ng / p.C_out, c = ng - phase * p.C_out;
    float v = Cs[m * (BN + 1) + n];
    if (p.groups > 0) {
      int pair = (m / p.L_out) * g_tile + n / cpg;
      v = (v - stats[pair * 2]) * stats[pair * 2 + 1];
      v = fmaf(v, __ldg(p.gn_gamma + c), __ldg(p.gn_beta + c));
    }
    v = apply_act(p.act, v);
    if (scale.present()) v *= scale.at(b, c);
    if (shift.present()) v += shift.at(b, c);
    if (p.res) {
      int rb = p.res_batch_mod > 0 ? b % p.res_batch_mod : b;
      v += ld_act(p.res, (int64_t)rb * p.res_bstride + (int64_t)l * p.res_lstride + c, p.res_dtype);
    }
    if (second_gemm) Cs[m * (BN + 1) + n] = v;
    else st_act(p.out, (int64_t)b * p.out_bstride + (int64_t)(l * p.phases + phase) * p.out_lstride + c, p.out_dtype, v);
  }
  if (!second_gemm) return;
  __syncthreads();

  // ---- 1x1 shortcut conv accumulated on top of the finished tile -------------------------------------
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;
  ConvSrc res_src{p.res_in, p.res_in_dtype, p.res_in_bstride, p.res_in_lstride, p.res_batch_mod, p.res_C, 1, 1, 0, p.L_out,
                  reinterpret_cast<const float*>(p.res_w)};
  gemm_mainloop<BN>(res_src, acc, As, Bs, st_b, st_l, n0, N_total);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int m = ty * 8 + i;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      int n = tx * TN + j, ng = n0 + n;
      float rb = (p.res_bias && ng < N_total) ? __ldg(p.res_bias + ng % p.C_out) : 0.f;
      Cs[m * (BN + 1) + n] += acc[i][j] + rb;
    }
  }
  __syncthreads();
  for (int idx = t; idx < kBM * BN; idx += kThreads) {
    int m = idx / BN, n = idx - m * BN;
    int r = row0 + m, ng = n0 + n;
    if (r >= rows || ng >= N_total) continue;
    int b = r / p.L_out, l = r - b * p.L_out;
    int phase = ng / p.C_out, c = ng - phase * p.C_out;
    st_act(p.out, (int64_t)b * p.out_bstride + (int64_t)(l * p.phases + phase) * p.out_lstride + c, p.out_dtype,
           Cs[m * (BN + 1) + n]);
  }
}

// choose the tile width; returns 0 if the op cannot be served by this kernel family
inline int conv_simt_pick_bn(const cds_conv_op& p) {
  int N = p.C_out * p.phases;
  if (p.groups > 0) {
    if (p.phases != 1 || p.C_out % p.groups != 0) return 0;
    if (p.L_out > kBM || (kBM % p.L_out) != 0) return 0;
    int cpg = p.C_out / p.groups;
    for (int bn : {32, 64, 128})
      if (bn % cpg == 0 && (bn >= N || bn >= 64)) return bn;
    for (int bn : {32, 64, 128})
      if (bn % cpg == 0) return bn;
    return 0;
  }
  if (N <= 32) return 32;
  if (N <= 64) return 64;
  return 128;
}

template <int BN>
inline cudaError_t conv_simt_launch_bn(const cds_conv_op& p, const int* iter_ptr, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_gemm_f32_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)ConvSmem<BN>::bytes);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  int rows = p.batch * p.L_out, N = p.C_out * p.phases;
  dim3 grid((rows + kBM - 1) / kBM, (N + BN - 1) / BN);
  conv_gemm_f32_kernel<BN><<<grid, kThreads, ConvSmem<BN>::bytes, st>>>(p, iter_ptr);
  return cudaGetLastError();
}

inline cudaError_t conv_simt_launch(const cds_conv_op& p, int bn, const int* iter_ptr, cudaStream_t st) {
  switch (bn) {
    case 32: return conv_simt_launch_bn<32>(p, iter_ptr, st);
    case 64: return conv_simt_launch_bn<64>(p, iter_ptr, st);
    case 128: return conv_simt_launch_bn<128>(p, iter_ptr, st);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace cds
