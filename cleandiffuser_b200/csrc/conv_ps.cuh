// CDS_OP_CONV, tensor-core path for SHORT sequences ("position-sliced" kernel): stride-1 Conv1d + GroupNorm + Mish
// (+ additive time row / identity residual / 1x1 shortcut conv) at a resolution of P = 4 positions -- the bottom of the
// UNets, where two thirds of JannerUNet1d's FLOPs live.
//
// conv_tc_kernel makes a 128-row tile out of 128/L whole trajectories and re-fetches the activation tile once per tap;
// at L = 4 that is 32 trajectories per weight slab and 5 x the activation bytes.  Here the GEMM rows are TRAJECTORIES:
//
//   D_l'[128 trajectories x N] (fp32, TMEM columns l'*N..)  +=  A_l[128 x KC] * W_(l - l' + pad)[N x KC]^T      |l - l'| <= pad
//
// * A_l = the activations of input position l: ONE TMA box {KC channels, 1 position, 128 trajectories} of the channels-last
//   bf16 tensor; every activation byte enters the SM once, the conv's zero padding is simply the absence of the
//   (l, l') pairs that fall outside [0, P) (14 MMAs instead of 20 for P = 4, taps = 5).
// * W_j = TMA box {KC, N} of the [tap][C_out][C_in] bf16 weight, fetched once per channel chunk and used by up to P MMAs:
//   4 x the trajectories per weight byte of conv_tc_kernel.
// * all P accumulators of a trajectory sit in the TMEM lane of ONE thread, so the GroupNorm statistics over
//   (P positions x C_out/8 channels) are plain in-thread sums: no shuffles.  Two passes over TMEM (statistics, then
//   normalise + Mish + store) keep the register footprint small; TMEM reads are cheap.
// * CTA tile = 128 trajectories x N = C_out/4 columns (2 GroupNorm groups: one per epilogue column slice); grid =
//   ceil(batch/128) x 4 CTAs (128 CTAs at batch 4096), one tile per CTA, 2-stage smem ring over the channel chunks,
//   warp roles as in conv_tc_kernel (8 epilogue warps, TMA producer, MMA issuer / TMEM owner).
//
// Algorithmic HBM bytes per launch: 2*(batch*P*C_in + batch*P*C_out) (+ shortcut input), weights once through L2.
#pragma once
#include "conv_tc.cuh"

namespace cds {

struct ConvPsParams {
  CUtensorMap tm_a, tm_b, tm_a2, tm_b2;
  CUtensorMap tm_out;             // output as a TMA-store target: box {16 channels, 1 position, 32 trajectories} (one epilogue warp's
  int out_tma;                    // lanes x 16 columns), staged in shared memory; valid when out_tma != 0
  // > 1: the n_tiles column-tile CTAs of a trajectory tile form a thread-block cluster of this size and share the activation
  // tiles -- CTA r fetches input position(s) l = r (mod cluster) once and MULTICASTS them into the shared memory of all of them
  // (each activation byte crosses the L2 -> SM fabric once per trajectory tile instead of once per column tile)
  int cluster;
  int batch, C_out, taps, pad;
  int kchunks, kchunks2;          // channel chunks of the main conv / of the shortcut conv
  int n_tiles;                    // column tiles per trajectory tile (C_out / N)
  int in_batch_mod, res_batch_mod;
  cds_vec bias, shift;
  const float* gn_gamma; const float* gn_beta; float gn_eps;
  const void* res; int64_t res_bstride; int res_lstride;
  const float* res_bias;
  void* out; int64_t out_bstride; int out_lstride;
  long long* trace;
};

// 16 epilogue warps (TMEM lane quarter = warp % 4, column slice = (warp / 4) % 2, position half = warp / 8), TMA producer
// (warp 16), MMA issuer / TMEM owner (warp 17).  The epilogue is MUFU/FMA-throughput work: 4 warps per scheduler overlap the
// two pipes far better than 2.
constexpr int kPsEpiWarps = 16;
constexpr int kPsEpiThreads = kPsEpiWarps * 32;
constexpr int kPsThreads = kPsEpiThreads + 64;
constexpr int kPsWarpTma = kPsEpiWarps, kPsWarpMma = kPsEpiWarps + 1;

template <int KC, int N, int P, bool HAS_RES>
struct ConvPsCfg {
  static constexpr int kTapsMax = 5;
  static constexpr int kRowBytes = KC * 2;
  static constexpr int kATile = 128 * kRowBytes;
  static constexpr int kBTile = N * kRowBytes;
  static constexpr int kStageBytes = P * kATile + kTapsMax * kBTile;
  static constexpr int kStages = KC == 64 ? 2 : 4;     // ~208 KB of operands in flight either way; finer chunks pipeline better
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024;
  static constexpr uint32_t kTmemCols = P * N * (HAS_RES ? 2 : 1);
  static_assert(kTmemCols == 128 || kTmemCols == 256 || kTmemCols == 512, "TMEM allocation must be a power of two <= 512");
  static_assert(kSmemBytes <= 227 * 1024, "stage ring does not fit");
};

// TF32: fp32 activations / weights read as TF32 (kind::tf32); KC stays the row width in bf16-equivalents (row bytes / 2), see
// conv_tc.cuh
template <int KC, int N, int P, bool HAS_RES, bool TF32>
__global__ void __launch_bounds__(kPsThreads, 1)
conv_ps_kernel(const __grid_constant__ ConvPsParams p, const int* __restrict__ iter_ptr) {
  using Cfg = ConvPsCfg<KC, N, P, HAS_RES>;
  constexpr int kStages = Cfg::kStages;
  constexpr int KE = TF32 ? KC / 2 : KC;            // channels per chunk
  constexpr int kActDtype = TF32 ? CDS_TF32 : CDS_BF16;      // output: fp32 storage rounded to TF32 / bf16
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[kStages];
  __shared__ __align__(8) uint64_t empty_bar[kStages];
  __shared__ __align__(8) uint64_t tmem_full_bar;
  __shared__ uint32_t tmem_base_holder;
  // per-column constants: 0 bias  1 GN gamma  2 GN beta  3 additive time row  4 shortcut bias
  __shared__ __align__(16) float s_col[5][N];
  __shared__ float2 s_part[2][2][128];             // GroupNorm partial (sum, sum of squares) [position half][column slice][trajectory]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - ptx::smem_u32(smem_raw));
  if (threadIdx.x == 0) { CDS_TRACE(0, gtimer()); CDS_TRACE(1, clock64()); }

  const int tile_b = blockIdx.x / p.n_tiles;          // trajectory tile
  const int n_off = (blockIdx.x % p.n_tiles) * N;     // first output channel of this CTA
  const int b0 = tile_b * 128;
  const int n_main = p.kchunks;
  const int n_chunks = n_main + (HAS_RES ? p.kchunks2 : 0);
  const uint32_t main_bytes = (uint32_t)(P * Cfg::kATile + p.taps * Cfg::kBTile);
  const uint32_t res_bytes = (uint32_t)(P * Cfg::kATile + Cfg::kBTile);

  const int cs = p.cluster;                           // cluster size (1 = no multicast)
  const uint32_t crank = cs > 1 ? ptx::cluster_ctarank() : 0u;
  const uint16_t cmask = (uint16_t)((1u << cs) - 1u);
  if (threadIdx.x == 0) {
    // a stage is free again when the MMAs of EVERY CTA of the cluster have consumed it (peers multicast into it)
    for (int s = 0; s < kStages; ++s) { ptx::mbar_init(&full_bar[s], 1); ptx::mbar_init(&empty_bar[s], (uint32_t)cs); }
    ptx::mbar_init(&tmem_full_bar, 1);
    ptx::fence_barrier_init();
  }
  if (warp == kPsWarpTma && lane == 0) {
    ptx::prefetch_tensormap(&p.tm_a);
    ptx::prefetch_tensormap(&p.tm_b);
    if (HAS_RES) { ptx::prefetch_tensormap(&p.tm_a2); ptx::prefetch_tensormap(&p.tm_b2); }
    if (p.out_tma) ptx::prefetch_tensormap(&p.tm_out);
  }
  if (warp == kPsWarpMma) ptx::tmem_alloc<Cfg::kTmemCols>(&tmem_base_holder);
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (cs > 1) ptx::cluster_sync();                    // every CTA's barriers exist before a peer can signal them
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = tmem_base_holder;
  if (threadIdx.x == 0) { CDS_TRACE(2, clock64()); ptx::grid_dep_launch_dependents(); }

  if (warp == kPsWarpTma) {
    // ===================================== TMA producer =====================================
    if (ptx::elect_one()) {
      auto load_w = [&](int c, int s) {               // weight tiles of chunk c into stage s
        uint8_t* sb = smem_al + s * Cfg::kStageBytes + P * Cfg::kATile;
        if (!HAS_RES || c < n_main) {
          for (int j = 0; j < p.taps; ++j)
            ptx::tma_load_2d(sb + (p.taps - 1 - j) * Cfg::kBTile, &p.tm_b, &full_bar[s], c * KE, j * p.C_out + n_off);   // slot = taps-1-j
        } else {
          ptx::tma_load_2d(sb, &p.tm_b2, &full_bar[s], (c - n_main) * KE, n_off);
        }
      };
      // weights do not depend on the previous kernel: arm the first ring fill and fetch them before the dependency wait
      const int pre = n_chunks < kStages ? n_chunks : kStages;
      for (int c = 0; c < pre; ++c) {
        ptx::mbar_expect_tx(&full_bar[c], (!HAS_RES || c < n_main) ? main_bytes : res_bytes);
        load_w(c, c);
      }
      ptx::grid_dep_wait();
      const int a_b0 = p.in_batch_mod > 0 ? b0 % p.in_batch_mod : b0;
      const int r_b0 = p.res_batch_mod > 0 ? b0 % p.res_batch_mod : b0;
      for (int c = 0; c < n_chunks; ++c) {
        const int s = c % kStages;
        const bool is_main = !HAS_RES || c < n_main;
        if (c >= pre) {
          ptx::mbar_wait(&empty_bar[s], ((c / kStages) & 1) ^ 1);
          ptx::mbar_expect_tx(&full_bar[s], is_main ? main_bytes : res_bytes);
          load_w(c, s);
        }
        uint8_t* sa = smem_al + s * Cfg::kStageBytes;
        for (int l = 0; l < P; ++l) {
          const void* tm = is_main ? (const void*)&p.tm_a : (const void*)&p.tm_a2;
          const int ck = is_main ? c * KE : (c - n_main) * KE, bb = is_main ? a_b0 : r_b0;
          if (cs == 1) ptx::tma_load_3d(sa + l * Cfg::kATile, tm, &full_bar[s], ck, l, bb);
          else if ((uint32_t)(l % cs) == crank) ptx::tma_load_3d_mc(sa + l * Cfg::kATile, tm, &full_bar[s], ck, l, bb, cmask);
        }
      }
      CDS_TRACE(8, clock64());
    }
  } else if (warp == kPsWarpMma) {
    // ===================================== MMA issuer =====================================
    if (ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc<TF32>(128, N);
      uint32_t started = 0;                           // bit l': accumulator D_l' has received its first MMA
      for (int c = 0; c < n_chunks; ++c) {
        const int s = c % kStages;
        ptx::mbar_wait(&full_bar[s], (c / kStages) & 1);
        ptx::tc_fence_after_sync();
        if (c == 0) CDS_TRACE(9, clock64());
        const uint32_t sa = smem_base + s * Cfg::kStageBytes;
        const uint32_t sb = sa + P * Cfg::kATile;
        if (!HAS_RES || c < n_main) {
          // The W tiles sit in REVERSED tap order (slot r = taps-1-j) and the accumulators D_l' in position order, so for one
          // input position l the valid outputs l' = lo..hi pair up with consecutive slots: ONE MMA of N' = (hi-lo+1)*N columns
          // instead of (hi-lo+1) MMAs of N columns -- small-N MMAs are bound by re-reading the A tile from shared memory
          // ((M+N)*32 B per K=16 step at 128 B/clk), N' >= 128 is tensor-bound.  The very first K step of the tile cannot
          // merge (the accumulate flag differs between already-started and fresh accumulators).
          for (int l = 0; l < P; ++l) {
            const uint64_t da = ptx::make_kmajor_desc<Cfg::kRowBytes>(sa + l * Cfg::kATile);
            const int lo = (l + p.pad - p.taps + 1) > 0 ? (l + p.pad - p.taps + 1) : 0;
            const int hi = (l + p.pad) < (P - 1) ? (l + p.pad) : (P - 1);
            const int slot0 = p.taps - 1 - (l - lo + p.pad);              // slot of the tap that feeds output position lo
            const uint64_t db = ptx::make_kmajor_desc<Cfg::kRowBytes>(sb + slot0 * Cfg::kBTile);
            const uint32_t idesc_m = ptx::make_idesc<TF32>(128, (hi - lo + 1) * N);
#pragma unroll
            for (int k = 0; k < KC / 16; ++k) {
              if (c == 0 && k == 0) {
                for (int lp = lo; lp <= hi; ++lp) {
                  const uint64_t dbj = ptx::make_kmajor_desc<Cfg::kRowBytes>(sb + (slot0 + lp - lo) * Cfg::kBTile);
                  ptx::umma<TF32>(tmem_base + (uint32_t)(lp * N), da, dbj, idesc, (started >> lp) & 1u);
                  started |= 1u << lp;
                }
              } else {
                ptx::umma<TF32>(tmem_base + (uint32_t)(lo * N), da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc_m, 1u);
              }
            }
          }
        } else {
          const uint64_t db = ptx::make_kmajor_desc<Cfg::kRowBytes>(sb);
#pragma unroll
          for (int l = 0; l < P; ++l) {
            const uint64_t da = ptx::make_kmajor_desc<Cfg::kRowBytes>(sa + l * Cfg::kATile);
#pragma unroll
            for (int k = 0; k < KC / 16; ++k)
              ptx::umma<TF32>(tmem_base + (uint32_t)(P * N + l * N), da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc,
                             (uint32_t)(c > n_main || k > 0));
          }
        }
        if (cs > 1) ptx::umma_commit_mc(&empty_bar[s], cmask); else ptx::umma_commit(&empty_bar[s]);
      }
      ptx::umma_commit(&tmem_full_bar);
    }
  } else {
    // ===================================== epilogue (warps 0..15) =====================================
    // thread = one trajectory (TMEM lane) x NH = N/2 columns (ONE GroupNorm group) x PH = P/2 positions; the two position
    // halves of a group exchange their partial statistics through shared memory.
    ptx::grid_dep_wait();
    const int iter = iter_ptr ? *iter_ptr : 0;
    constexpr int NH = N / 2;
    static_assert(NH == 16 || NH == 32, "one GroupNorm group of 16 or 32 channels per epilogue column slice");
    const int q = warp & 3, half = (warp >> 2) & 1, ph = warp >> 3;
    constexpr int PH = P / 2;
    const int lp0 = ph * PH;                          // first position of this thread
    {
      const float* bstep = p.bias.step ? p.bias.step + (int64_t)iter * p.bias.step_stride : nullptr;
      const float* hstep = p.shift.step ? p.shift.step + (int64_t)iter * p.shift.step_stride : nullptr;
      for (int n = threadIdx.x; n < N; n += kPsEpiThreads) {
        const int c = n_off + n;
        s_col[0][n] = bstep ? __ldg(bstep + c) - group_mean(bstep, c - c % NH, NH) : 0.f;   // (a group = NH = C_out / 8 columns)
        s_col[1][n] = __ldg(p.gn_gamma + c);
        s_col[2][n] = __ldg(p.gn_beta + c);
        s_col[3][n] = hstep ? __ldg(hstep + c) : 0.f;
        s_col[4][n] = (HAS_RES && p.res_bias) ? __ldg(p.res_bias + c) : 0.f;
      }
      ptx::named_bar_sync(1, kPsEpiThreads);
    }
    const int b = b0 + 32 * q + lane;
    const bool valid = b < p.batch;
    const int col0 = half * NH;                       // CTA-tile column of this thread's slice
    const uint32_t t_row = tmem_base + ((uint32_t)(32 * q) << 16);
    const int rb = p.res_batch_mod > 0 ? b % p.res_batch_mod : b;

    ptx::mbar_wait(&tmem_full_bar, 0);
    ptx::tc_fence_after_sync();
    if (threadIdx.x == 0) CDS_TRACE(10, clock64());

    // ---- pass 1: GroupNorm statistics of (accumulator + bias) over P positions x NH channels, all in this thread.
    // TMEM reads are double-buffered: the load of the next position is in flight while this one is summed.
    float s1 = 0.f, s2 = 0.f;
    {
      float va[NH], vb[NH];
      ptx::tmem_ld_nowait<NH>(t_row + (uint32_t)(lp0 * N + col0), va);
      auto accumulate = [&](const float (&v)[NH]) {
#pragma unroll
        for (int k = 0; k < NH / 4; ++k) {
          const float4 bb = reinterpret_cast<const float4*>(&s_col[0][col0])[k];
          const float x0 = v[4 * k] + bb.x, x1 = v[4 * k + 1] + bb.y, x2 = v[4 * k + 2] + bb.z, x3 = v[4 * k + 3] + bb.w;
          s1 += (x0 + x1) + (x2 + x3);
          s2 = fmaf(x0, x0, s2); s2 = fmaf(x1, x1, s2); s2 = fmaf(x2, x2, s2); s2 = fmaf(x3, x3, s2);
        }
      };
      static_assert(PH == 2, "pass 1 ping-pongs two register buffers over the two positions of this thread");
      ptx::tmem_ld_wait();
      ptx::tmem_ld_nowait<NH>(t_row + (uint32_t)((lp0 + 1) * N + col0), vb);
      accumulate(va);
      ptx::tmem_ld_wait();
      accumulate(vb);
    }
    // first chunk of pass 2 is already on its way while the halves exchange their partial sums
    float vbuf[2][16];
    ptx::tmem_ld_nowait<16>(t_row + (uint32_t)(lp0 * N + col0), vbuf[0]);
    s_part[ph][half][32 * q + lane] = make_float2(s1, s2);
    ptx::named_bar_sync(1, kPsEpiThreads);
    { const float2 o2 = s_part[ph ^ 1][half][32 * q + lane]; s1 += o2.x; s2 += o2.y; }
    const float inv_cnt = 1.f / (float)(P * NH);
    const float mean = s1 * inv_cnt;
    const float ga = rsqrt_ftz(fmaxf(fmaf(s2, inv_cnt, -mean * mean), 0.f) + p.gn_eps);
    const float gc = -mean * ga;

    // ---- pass 2: normalise, affine, Mish, additive terms, store; 16-column chunks, the next chunk's TMEM read in flight
    const bool add_res = p.res != nullptr;
    constexpr int kChunks = PH * (NH / 16);
#pragma unroll
    for (int ci = 0; ci < kChunks; ++ci) {
      const int lp = lp0 + ci / (NH / 16), h = ci % (NH / 16);
      const int n0 = col0 + 16 * h;                   // CTA-tile column
      float (&v)[16] = vbuf[ci & 1];
      float addv[16];
      const float4* sh4 = reinterpret_cast<const float4*>(&s_col[3][n0]);
#pragma unroll
      for (int k = 0; k < 4; ++k) { const float4 s = sh4[k]; addv[4 * k] = s.x; addv[4 * k + 1] = s.y; addv[4 * k + 2] = s.z; addv[4 * k + 3] = s.w; }
      if (add_res) {
        float resv[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) resv[j] = 0.f;
        if (valid) load_row<16>(p.res, (int64_t)rb * p.res_bstride + (int64_t)lp * p.res_lstride + n_off + n0, kActDtype, resv);
#pragma unroll
        for (int j = 0; j < 16; ++j) addv[j] += resv[j];
      }
      ptx::tmem_ld_wait();
      if (ci + 1 < kChunks) {
        const int lp1 = lp0 + (ci + 1) / (NH / 16), h1 = (ci + 1) % (NH / 16);
        ptx::tmem_ld_nowait<16>(t_row + (uint32_t)(lp1 * N + col0 + 16 * h1), vbuf[(ci + 1) & 1]);
      }
      if constexpr (HAS_RES) {
        float r2[16];
        ptx::tmem_ld<16>(t_row + (uint32_t)(P * N + lp * N + n0), r2);      // (its wait also completes the prefetch above)
        const float4* rb4 = reinterpret_cast<const float4*>(&s_col[4][n0]);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float4 s = rb4[k];
          addv[4 * k] += r2[4 * k] + s.x; addv[4 * k + 1] += r2[4 * k + 1] + s.y;
          addv[4 * k + 2] += r2[4 * k + 2] + s.z; addv[4 * k + 3] += r2[4 * k + 3] + s.w;
        }
      }
      const float4* b4 = reinterpret_cast<const float4*>(&s_col[0][n0]);
      const float4* ga4 = reinterpret_cast<const float4*>(&s_col[1][n0]);
      const float4* be4 = reinterpret_cast<const float4*>(&s_col[2][n0]);
      float o[16];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float4 bb = b4[k], gm = ga4[k], be = be4[k];
        o[4 * k + 0] = mish_fma(fmaf(fmaf(v[4 * k + 0] + bb.x, ga, gc), gm.x, be.x), addv[4 * k + 0]);
        o[4 * k + 1] = mish_fma(fmaf(fmaf(v[4 * k + 1] + bb.y, ga, gc), gm.y, be.y), addv[4 * k + 1]);
        o[4 * k + 2] = mish_fma(fmaf(fmaf(v[4 * k + 2] + bb.z, ga, gc), gm.z, be.z), addv[4 * k + 2]);
        o[4 * k + 3] = mish_fma(fmaf(fmaf(v[4 * k + 3] + bb.w, ga, gc), gm.w, be.w), addv[4 * k + 3]);
      }
      if (p.out_tma) {
        // 32 trajectories (lanes) x 16 columns of position lp through shared memory and ONE bulk store: a warp-level st.global
        // would touch 32 cache lines per instruction.  The operand ring is idle once the accumulators are complete (one tile
        // per CTA), its first 2 KB (fp32) / 1 KB (bf16) per warp serve as staging rows in the swizzle of tm_out.
        uint8_t* const stg = smem_al + warp * 2048;
        if (lane == 0) ptx::bulk_wait_group_read<0>();
        __syncwarp();
        if constexpr (TF32) {
          uint8_t* const sr = stg + lane * 64;
#pragma unroll
          for (int k = 0; k < 4; ++k)
            *reinterpret_cast<float4*>(sr + ((k ^ ((lane >> 1) & 3)) << 4)) =
                make_float4(round_tf32(o[4 * k]), round_tf32(o[4 * k + 1]), round_tf32(o[4 * k + 2]), round_tf32(o[4 * k + 3]));
        } else {
          uint8_t* const sr = stg + lane * 32;
          const int sw = (lane >> 2) & 1;
          uint32_t w[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) { __nv_bfloat162 h2 = __floats2bfloat162_rn(o[2 * k], o[2 * k + 1]); w[k] = *reinterpret_cast<uint32_t*>(&h2); }
          *reinterpret_cast<uint4*>(sr + ((0 ^ sw) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
          *reinterpret_cast<uint4*>(sr + ((1 ^ sw) << 4)) = make_uint4(w[4], w[5], w[6], w[7]);
        }
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          ptx::tma_store_3d(&p.tm_out, stg, n_off + n0, lp, b0 + 32 * q);
          ptx::bulk_commit_group();
        }
      } else if (valid) {
        store_row<16>(p.out, (int64_t)b * p.out_bstride + (int64_t)lp * p.out_lstride + n_off + n0, kActDtype, o);
      }
    }
    if (lane == 0) ptx::bulk_wait_group<0>();        // the bulk stores are complete before the CTA retires
    if (threadIdx.x == 0) { CDS_TRACE(11, clock64()); CDS_TRACE(5, 1LL); }
    ptx::tc_fence_before_sync();
  }

  __syncthreads();
  if (cs > 1) ptx::cluster_sync();                    // no CTA retires while a peer may still multicast into it / signal its barriers
  if (warp == kPsWarpMma) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
  if (threadIdx.x == 0) { CDS_TRACE(3, clock64()); CDS_TRACE(4, gtimer()); }
}

// ------------------------------------------------------------------------------------------------ host side
constexpr int kPsPositions = 4;
constexpr int kPsKC = 32;            // channel chunk: 32 (SWIZZLE_64B tiles, 4-stage ring) pipelines better than 64 (2 stages)

// CTA tile width: a quarter of the layer (two GroupNorm groups); 0 = the kernel is not instantiated for this layer
inline int conv_ps_width(const cds_conv_op& c) {
  if (c.C_out == 256) return 64;
  if (c.C_out == 128) return 32;
  return 0;
}

// Can the position-sliced kernel serve this op?  (a subset of conv_tc_eligible: same layouts, same weight packing)
inline bool conv_ps_eligible(const cds_conv_op& c) {
  if (!conv_tc_eligible(c)) return false;
  if (c.L_in != kPsPositions || c.L_out != kPsPositions || c.stride != 1 || c.phases != 1) return false;
  if (c.taps < 1 || c.taps > 5 || (c.taps & 1) == 0 || c.pad != c.taps / 2) return false;
  if (c.groups != 8 || c.act != CDS_ACT_MISH || conv_ps_width(c) == 0) return false;
  if (c.C_in % 64 != 0 || (c.res_w && c.res_C % 64 != 0)) return false;
  if (c.bias.sample || c.scale.step || c.scale.sample || c.shift.sample) return false;
  if (conv_is_tf32(c)) { if (c.out_dtype != CDS_TF32 || (c.res && c.res_dtype == CDS_BF16)) return false; }
  else if (c.out_dtype != CDS_BF16 || (c.res && c.res_dtype != CDS_BF16)) return false;
  if (c.in_batch_mod > 0 && c.in_batch_mod % 128 != 0) return false;
  if (c.res_batch_mod > 0 && c.res_batch_mod % 128 != 0) return false;
  const char* env = getenv("CDS_PS");
  if (env && env[0] == '0') return false;
  return true;
}

struct ConvPsLaunch {
  ConvPsParams prm;
  bool tf32 = false;
  int n = 0;
  bool has_res = false;
  dim3 grid;
};

inline bool conv_ps_prepare(const cds_conv_op& c, ConvPsLaunch* out) {
  ConvPsLaunch& L = *out;
  memset(&L.prm, 0, sizeof(L.prm));
  ConvPsParams& p = L.prm;
  constexpr int kc = kPsKC;
  const bool tf32 = conv_is_tf32(c);
  const int ke = tf32 ? kc / 2 : kc;
  L.tf32 = tf32;
  L.n = conv_ps_width(c);
  L.has_res = c.res_w != nullptr;
  const uint64_t in_b = c.in_batch_mod > 0 ? (uint64_t)c.in_batch_mod : (uint64_t)c.batch;
  {
    uint64_t dims[3] = {(uint64_t)c.C_in, (uint64_t)c.L_in, in_b};
    uint64_t str[2] = {(uint64_t)c.in_lstride, (uint64_t)c.in_bstride};
    uint32_t box[3] = {(uint32_t)ke, 1u, 128u};
    if (!encode_act_map(&p.tm_a, c.in, 3, dims, str, box, kc, tf32)) return false;
  }
  {
    uint64_t dims[2] = {(uint64_t)c.C_in, (uint64_t)c.taps * c.C_out};
    uint64_t str[1] = {(uint64_t)c.C_in};
    uint32_t box[2] = {(uint32_t)ke, (uint32_t)L.n};
    if (!encode_act_map(&p.tm_b, c.w, 2, dims, str, box, kc, tf32)) return false;
  }
  if (L.has_res) {
    const uint64_t r_b = c.res_batch_mod > 0 ? (uint64_t)c.res_batch_mod : (uint64_t)c.batch;
    uint64_t dims[3] = {(uint64_t)c.res_C, (uint64_t)c.L_out, r_b};
    uint64_t str[2] = {(uint64_t)c.res_in_lstride, (uint64_t)c.res_in_bstride};
    uint32_t box[3] = {(uint32_t)ke, 1u, 128u};
    if (!encode_act_map(&p.tm_a2, c.res_in, 3, dims, str, box, kc, tf32)) return false;
    uint64_t d2[2] = {(uint64_t)c.res_C, (uint64_t)c.C_out};
    uint64_t s2[1] = {(uint64_t)c.res_C};
    uint32_t b2[2] = {(uint32_t)ke, (uint32_t)L.n};
    if (!encode_act_map(&p.tm_b2, c.res_w, 2, d2, s2, b2, kc, tf32)) return false;
  }
  p.batch = c.batch; p.C_out = c.C_out; p.taps = c.taps; p.pad = c.pad;
  p.kchunks = c.C_in / ke; p.kchunks2 = L.has_res ? c.res_C / ke : 0;
  p.n_tiles = c.C_out / L.n;
  p.in_batch_mod = c.in_batch_mod; p.res_batch_mod = c.res_batch_mod;
  p.bias = c.bias; p.shift = c.shift;
  p.gn_gamma = c.gn_gamma; p.gn_beta = c.gn_beta; p.gn_eps = c.gn_eps;
  p.res = c.res; p.res_bstride = c.res_bstride; p.res_lstride = c.res_lstride; p.res_bias = c.res_bias;
  p.out = c.out; p.out_bstride = c.out_bstride; p.out_lstride = c.out_lstride;
  {
    const int oes = tf32 ? 4 : 2;
    p.out_tma = 0;
    PFN_encodeTiled enc = get_encode_tiled();
    const bool ok = ((uintptr_t)c.out % 16) == 0 && ((int64_t)c.out_lstride * oes) % 16 == 0 && ((int64_t)c.out_bstride * oes) % 16 == 0 &&
                    !getenv("CDS_NO_TMA_STORE");
    cuuint64_t gdim[3] = {(cuuint64_t)c.C_out, (cuuint64_t)c.L_out, (cuuint64_t)c.batch};
    cuuint64_t gstr[2] = {(cuuint64_t)c.out_lstride * oes, (cuuint64_t)c.out_bstride * oes};
    cuuint32_t bx[3] = {16u, 1u, 32u};
    cuuint32_t es[3] = {1u, 1u, 1u};
    if (ok && enc && enc(&p.tm_out, tf32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, c.out, gdim, gstr, bx, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, tf32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B,
                         CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
      p.out_tma = 1;
  }
  L.grid = dim3((unsigned)(((c.batch + 127) / 128) * p.n_tiles));
  // column-tile CTAs of a trajectory tile are consecutive blocks: one cluster per trajectory tile.  Opt-in (CDS_MULTICAST=1):
  // measured slower than unicast on B200 (see conv_tc_prepare)
  { const char* mc = getenv("CDS_MULTICAST"); p.cluster = (p.n_tiles == 4 && kPsPositions % 4 == 0 && mc && mc[0] == '1') ? 4 : 1; }
  return true;
}

template <int N, bool HAS_RES, bool TF32>
cudaError_t conv_ps_launch_t(const ConvPsLaunch& L, const int* iter_ptr, cudaStream_t st) {
  using Cfg = ConvPsCfg<kPsKC, N, kPsPositions, HAS_RES>;
  static bool attr = false;
  static bool pdl = true;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(conv_ps_kernel<kPsKC, N, kPsPositions, HAS_RES, TF32>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
    if (e != cudaSuccess) return e;
    if (getenv("CDS_DEBUG"))
      fprintf(stderr, "[cds] conv_ps<%d,%d,%d,%d,%s>: smem %d B, tmem %u columns\n", kPsKC, N, kPsPositions, (int)HAS_RES,
              TF32 ? "tf32" : "bf16", Cfg::kSmemBytes, Cfg::kTmemCols);
    const char* pdl_env = getenv("CDS_PDL");
    pdl = !(pdl_env && pdl_env[0] == '0');
    attr = true;
  }
  ConvPsParams prm = L.prm;
  prm.trace = conv_tc_trace_hook((int)L.grid.x);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = L.grid; cfg.blockDim = dim3(kPsThreads); cfg.dynamicSmemBytes = Cfg::kSmemBytes; cfg.stream = st;
  cudaLaunchAttribute at[2];
  int na = 0;
  if (pdl) { at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[na].val.programmaticStreamSerializationAllowed = 1; ++na; }
  if (prm.cluster > 1) {
    at[na].id = cudaLaunchAttributeClusterDimension;
    at[na].val.clusterDim.x = (unsigned)prm.cluster; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
    ++na;
  }
  cfg.attrs = at; cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, conv_ps_kernel<kPsKC, N, kPsPositions, HAS_RES, TF32>, prm, iter_ptr);
}
template <int N, bool HAS_RES, bool TF32>
cudaError_t conv_ps_preload_t() {
  cudaFuncAttributes a;
  return cudaFuncGetAttributes(&a, conv_ps_kernel<kPsKC, N, kPsPositions, HAS_RES, TF32>);
}

// X(N, HAS_RES, TF32) over every instantiation
#define CDS_PS_VARIANTS(X)                                                                   \
  X(32, false, false) X(32, true, false) X(64, false, false) X(64, true, false)             \
  X(32, false, true) X(32, true, true) X(64, false, true) X(64, true, true)

#ifndef CDS_PS_INSTANTIATE
#define CDS_PS_EXTERN(N_, R_, T_)                                                                                 \
  extern template cudaError_t conv_ps_launch_t<N_, R_, T_>(const ConvPsLaunch&, const int*, cudaStream_t);        \
  extern template cudaError_t conv_ps_preload_t<N_, R_, T_>();
CDS_PS_VARIANTS(CDS_PS_EXTERN)
#undef CDS_PS_EXTERN

inline cudaError_t conv_ps_launch(const ConvPsLaunch& L, const int* iter_ptr, cudaStream_t st) {
#define CDS_PS_CASE(N_, R_, T_) if (L.n == N_ && L.has_res == R_ && L.tf32 == T_) return conv_ps_launch_t<N_, R_, T_>(L, iter_ptr, st);
  CDS_PS_VARIANTS(CDS_PS_CASE)
#undef CDS_PS_CASE
  return cudaErrorInvalidValue;
}
inline cudaError_t conv_ps_preload_all() {
  cudaError_t e;
#define CDS_PS_PRE(N_, R_, T_) if ((e = conv_ps_preload_t<N_, R_, T_>()) != cudaSuccess) return e;
  CDS_PS_VARIANTS(CDS_PS_PRE)
#undef CDS_PS_PRE
  return cudaSuccess;
}
#endif

}  // namespace cds
