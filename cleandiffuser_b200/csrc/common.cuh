// Shared device helpers for libcds (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "cds.h"

namespace cds {

// vec(b, c) = step[iter*step_stride + c] + sample[b*sample_stride + c]
struct VecRef {
  const float* step;
  const float* sample;
  int64_t sample_stride;
  __device__ __forceinline__ bool present() const { return step != nullptr || sample != nullptr; }
  __device__ __forceinline__ float at(int b, int c) const {
    float v = 0.f;
    if (step) v = __ldg(step + c);
    if (sample) v += __ldg(sample + (int64_t)b * sample_stride + c);
    return v;
  }
};

__device__ __forceinline__ VecRef resolve(const cds_vec& v, int iter) {
  VecRef r;
  r.step = v.step ? v.step + (int64_t)iter * v.step_stride : nullptr;
  r.sample = v.sample;
  r.sample_stride = v.sample_stride;
  return r;
}

// mean of v[first .. first + n).  The tensor-core kernels subtract it from the bias of a GroupNorm group when they stage the
// per-column constants: GroupNorm does not change under a common shift of its group, and with the group's common offset gone
// the single-pass moments E[y^2] - E[y]^2 in fp32 no longer cancel (a bias of 256 group sigmas cost ~1e-2 in rstd).  Every
// column of a group sums the same values in the same order, so the shift is bit-identical across the group.
__device__ __forceinline__ float group_mean(const float* v, int first, int n) {
  float s = 0.f;
  for (int j = 0; j < n; ++j) s += __ldg(v + first + j);
  return s / (float)n;
}

// activations; formulas follow ATen's fp32 CUDA/CPU definitions
__device__ __forceinline__ float act_mish(float x) {
  // x * tanh(softplus(x)), softplus with torch's threshold of 20
  float sp = x > 20.f ? x : log1pf(expf(x));
  return x * tanhf(sp);
}
__device__ __forceinline__ float act_silu(float x) { return x / (1.f + expf(-x)); }
__device__ __forceinline__ float act_gelu_tanh(float x) {
  const float kBeta = 0.7978845608028654f;  // sqrt(2/pi)
  const float kKappa = 0.044715f;
  float inner = kBeta * (x + kKappa * x * x * x);
  return 0.5f * x * (1.f + tanhf(inner));
}
__device__ __forceinline__ float apply_act(int act, float x) {
  switch (act) {
    case CDS_ACT_MISH: return act_mish(x);
    case CDS_ACT_SILU: return act_silu(x);
    case CDS_ACT_GELU_TANH: return act_gelu_tanh(x);
    case CDS_ACT_MISH_SILU: return act_silu(act_mish(x));
    case CDS_ACT_LEAKY_RELU: return x > 0.f ? x : 0.01f * x;
    case CDS_ACT_GELU_ERF: return 0.5f * x * (1.f + erff(x * 0.7071067811865476f));
    default: return x;
  }
}

// fp32 -> nearest TF32-representable fp32 (ties away from zero): two integer ops
__device__ __forceinline__ float round_tf32(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }
// value as an operator stores it into a tensor of cds_dtype `dtype` (fp32 storage: CDS_F32 as is, CDS_TF32 rounded)
__device__ __forceinline__ float f32_for_store(float x, int dtype) { return dtype == CDS_TF32 ? round_tf32(x) : x; }

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

}  // namespace cds
