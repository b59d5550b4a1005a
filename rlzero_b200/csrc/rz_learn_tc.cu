// rlzero_b200 -- the training step of the 128-channel ResNet trunk on the tensor cores.
//
// Reference op: AlphaZeroAgent.learn (rlzero/games/gomoku/alphazero_agent.py:59-86) -- loss.backward() +
// optimizer.step() -- for the ResNet-N policy-value net of SURVEY.md section 7 (conv3x3 + BatchNorm2d in training
// mode + skip + ReLU).  Activations and gradients travel as bf16 in the padded position layout of the inference path
// ([board*S*S + y*S + x][128 channels], zero at x >= W / y >= H and in the tail rows up to the multiple of 256 rows),
// statistics, reductions and parameter gradients are fp32.  The row stride S is 16 for boards up to 15x15 and 20 for
// 16x16 .. 19x19 (the Go boards of config 4); the _ex entry points take it, the plain ones are their S = 16 calls.
//
//   forward convolution   rz_net_conv3x3_tc2 (rz_net_tc2.cu) at S = 16, rz_net_conv3x3_tc3 (rz_net_tc3.cu) at S = 20,
//                         raw output (bias, no ReLU)
//   data gradient         the SAME kernel with the weights transposed and the taps mirrored (rz_learn_pack_conv_tc)
//   weight gradient       rz_conv_wgrad_tc_kernel below: dW[tap][co][ci] = sum_p dy[p][co] * x[p + d(tap)][ci], a
//                         GEMM whose reduction runs over the POSITIONS.  Both operands are stored position-major
//                         (the reduction index is the row), i.e. they are "MN-major" UMMA operands: the 128-byte-swizzled
//                         tiles TMA writes -- 64 channels = 128 B per row -- are exactly the canonical MN-major
//                         SWIZZLE_128B atoms (8 rows x 128 B, 1024 B apart along K, the other 64 channels LBO apart),
//                         so no transpose is ever materialised; the 9 taps are row-shifted descriptors on one halo tile
//                         of x, as in the forward kernel.  fp32 accumulators stay in TMEM for the whole launch (3 taps
//                         x 128 columns per CTA); CTAs form triples (one per filter row) that walk the same position
//                         tiles, so HBM sees each tile once and L2 serves the other two.  Templated on S: an (S + 1)-row
//                         halo, filter rows S rows apart; at S = 20 a tile may straddle two boards (pad squares are 0).
//   stem                  forward: the inference stem fed from float32 planes (4 planes, or the 17 of GoEnv.observe);
//                         weight gradient: the kernel above with the planes as channels 0 .. P-1 of a tile
//   BatchNorm             batch statistics / normalise + skip + ReLU / the two backward reductions / the backward
//                         apply as row-parallel kernels (a warp owns a row of 128 channels = 256 B).
#include <cuda_bf16.h>

#include "rz_common.cuh"
#include "rz_tc.cuh"

namespace {

// ---------------------------------------------------------------------------------------------------------
// weight gradient on tcgen05
// ---------------------------------------------------------------------------------------------------------
constexpr int WG_TILE = 128;                        // positions per tile (the K extent of one stage)
constexpr int WG_DY_HALF = WG_TILE * 128;           // 16384 B: [128 rows][64 channels]
constexpr int WG_STAGES = 3;
constexpr int WG_THREADS = 192;                     // producer warp, MMA warp, 4 drain warps

// the stage geometry of row stride S: x tiles carry an (S + 1)-row halo on each side
//   S = 16: 162-row x tiles, stages of 74240 B, 224768 B of shared memory
//   S = 20: 170-row x tiles, stages of 76288 B, 230912 B (the 232448 B limit allows no fourth stage at either stride)
template <int kS>
struct WgGeo {
  static constexpr int HALO = kS + 1;
  static constexpr int XROWS = WG_TILE + 2 * HALO;
  static constexpr int X_HALF = XROWS * 128;
  static constexpr int STAGE = 2 * WG_DY_HALF + 2 * X_HALF;
  static constexpr int CTRL = WG_STAGES * STAGE;
  static constexpr int SMEM = CTRL + 1024 + 1024;   // + control block + alignment slack
};

// MN-major SWIZZLE_128B operand: start address, LBO = byte distance between the two 64-channel halves, SBO = 1024 B
// between 8-row groups along K (cute::UMMA::make_umma_desc<Major::MN> for Layout_MN_SW128_Atom)
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)(1024u >> 4) << 32;
  d |= (uint64_t)1 << 46;                            // descriptor version 1 (sm_100)
  d |= (uint64_t)2 << 61;                            // SWIZZLE_128B
  return d;
}
// kind::f16 instruction descriptor: D = f32, A = B = bf16, both operands MN-major (bits 15 / 16), M x N
__host__ __device__ constexpr uint32_t umma_idesc_bf16_mn(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

struct WgradParams {
  float* part;        // [n_splits][9][128 co][128 ci]
  int n_tiles;        // 128-row tiles of the position layout
  int n_splits;
};

template <int kS>
__global__ void __launch_bounds__(WG_THREADS, 1)
rz_conv_wgrad_tc_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_dy,
                        const WgradParams p) {
  using G = WgGeo<kS>;
  static_assert(G::SMEM <= 232448, "shared memory budget");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (rz::smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* al = smem_raw + (base - rz::smem_u32(smem_raw));
  const uint32_t ctrl = base + G::CTRL;
  const uint32_t bar_full = ctrl, bar_empty = ctrl + 32, bar_done = ctrl + 64;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(al + G::CTRL + 96);
  const int warp = rz::uniform_i32((int)(threadIdx.x >> 5)), lane = threadIdx.x & 31;
  const int split = blockIdx.x / 3, row_grp = blockIdx.x % 3;       // filter row dy = row_grp - 1

  if (threadIdx.x == 0) {
    rz::tma_prefetch_desc(&tmap_x);
    rz::tma_prefetch_desc(&tmap_dy);
    for (int s = 0; s < WG_STAGES; ++s) { rz::mbar_init(bar_full + 8 * s, 1); rz::mbar_init(bar_empty + 8 * s, 1); }
    rz::mbar_init(bar_done, 1);
    rz::fence_barrier_init();
  }
  if (warp == 1) { rz::tmem_alloc(rz::smem_u32(tmem_holder), 512); rz::tmem_relinquish(); }
  rz::tc_fence_before();
  __syncthreads();
  rz::tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  const int n_my = split < p.n_tiles ? (p.n_tiles - split + p.n_splits - 1) / p.n_splits : 0;

  if (warp == 0) {
    if (lane == 0) {
      for (int it = 0; it < n_my; ++it) {
        const int st = it % WG_STAGES;
        rz::mbar_wait(bar_empty + 8 * st, ((uint32_t)(it / WG_STAGES) & 1u) ^ 1u);
        rz::mbar_expect_tx(bar_full + 8 * st, (uint32_t)G::STAGE);
        const int row0 = (split + it * p.n_splits) * WG_TILE;
        const uint32_t sb = base + (uint32_t)st * G::STAGE;
        for (int h = 0; h < 2; ++h) {
          rz::tma_load_2d(sb + (uint32_t)h * WG_DY_HALF, &tmap_dy, bar_full + 8 * st, h * 64, row0);
          rz::tma_load_2d(sb + 2u * WG_DY_HALF + (uint32_t)h * G::X_HALF, &tmap_x, bar_full + 8 * st, h * 64, row0 - G::HALO);
        }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = umma_idesc_bf16_mn(128, 128);
    const uint32_t issue = rz::elect_one();
    const uint32_t tmem_u = rz::uniform_u32(tmem_base);
    for (int it = 0; it < n_my; ++it) {
      const int st = it % WG_STAGES;
      rz::mbar_wait(bar_full + 8 * st, (uint32_t)(it / WG_STAGES) & 1u);
      rz::tc_fence_after();
      const uint32_t dyb = base + (uint32_t)st * G::STAGE, xb = dyb + 2u * WG_DY_HALF;
#pragma unroll 1
      for (int t = 0; t < 3; ++t) {
        const int shift = G::HALO + (row_grp - 1) * kS + (t - 1);        // rows into the halo tile of x
#pragma unroll
        for (int ks = 0; ks < WG_TILE / 16; ++ks) {
          const uint64_t adesc = umma_desc_mn_sw128(dyb + (uint32_t)ks * 2048u, WG_DY_HALF);
          const uint64_t bdesc = umma_desc_mn_sw128(xb + (uint32_t)(shift + ks * 16) * 128u, G::X_HALF);
          rz::umma_bf16_pred(tmem_u + (uint32_t)(t * 128), adesc, bdesc, idesc, (it > 0 || ks > 0) ? 1u : 0u, issue);
        }
      }
      rz::umma_commit_pred(bar_empty + 8 * st, issue);      // the stage may be refilled once these MMAs have read it
    }
    rz::umma_commit_pred(bar_done, issue);
  } else {
    // drain: TMEM lane = output channel co, column = input channel ci -> part[split][tap][co][ci]
    rz::mbar_wait(bar_done, 0);
    rz::tc_fence_after();
    const int q = warp & 3;
    const int co = q * 32 + lane;
    for (int t = 0; t < 3; ++t) {
      float* out = p.part + (((size_t)split * 9 + (size_t)(row_grp * 3 + t)) * 128 + co) * 128;
#pragma unroll 1
      for (int ch = 0; ch < 4; ++ch) {
        uint32_t acc[32];
        if (n_my > 0) {
          rz::tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(t * 128 + ch * 32), acc);
          rz::tmem_ld_wait();
        } else {
#pragma unroll
          for (int e = 0; e < 32; ++e) acc[e] = 0u;
        }
#pragma unroll
        for (int e = 0; e < 32; e += 4)
          *reinterpret_cast<uint4*>(out + ch * 32 + e) = make_uint4(acc[e], acc[e + 1], acc[e + 2], acc[e + 3]);
      }
    }
  }
  rz::tc_fence_before();
  __syncthreads();
  if (warp == 1) { rz::tc_fence_after(); rz::tmem_dealloc(tmem_base, 512); }
}

// dw[co][ci][tap] = sum_s part[s][tap][co][ci]
__global__ void rz_wgrad_tc_final_kernel(const float* __restrict__ part, float* __restrict__ dw, int n_splits) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;       // over [tap][co][ci]
  if (i >= 9 * 128 * 128) return;
  const int ci = i & 127, co = (i >> 7) & 127, tap = i >> 14;
  float t = 0.0f;
  for (int s = 0; s < n_splits; ++s) t += part[(size_t)s * (9 * 128 * 128) + i];
  dw[((size_t)co * 128 + ci) * 9 + tap] = t;
}

// ---------------------------------------------------------------------------------------------------------
// weights: fp32 [128][128][3][3] -> bf16 forward [tap][co][ci] and data-gradient [8 - tap][ci][co]
// ---------------------------------------------------------------------------------------------------------
__global__ void rz_pack_conv_tc_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wf,
                                       __nv_bfloat16* __restrict__ wb) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 128 * 128 * 9) return;
  const int tap = i % 9, ci = (i / 9) & 127, co = i / (9 * 128);
  const __nv_bfloat16 v = __float2bfloat16_rn(w[i]);
  wf[((size_t)tap * 128 + co) * 128 + ci] = v;
  wb[((size_t)(8 - tap) * 128 + ci) * 128 + co] = v;
}
// inference weights of a 128 -> 128 trunk layer straight from the float32 parameters: eval-mode BatchNorm folded in
// (float64 arithmetic, like the host packing of NativeForward.refresh_weights), bf16 [tap][cout][cin] + fp32 bias
__global__ void rz_pack_conv_bn_tc_kernel(const float* __restrict__ w, const float* __restrict__ cbias,
                                          const float* __restrict__ gamma, const float* __restrict__ beta,
                                          const float* __restrict__ mean, const float* __restrict__ var, float eps,
                                          __nv_bfloat16* __restrict__ wout, float* __restrict__ bout) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 128 * 128 * 9) return;
  const int tap = i % 9, ci = (i / 9) & 127, co = i / (9 * 128);
  double sc = 1.0;
  if (gamma) sc = (double)gamma[co] / sqrt((double)var[co] + (double)eps);
  wout[((size_t)tap * 128 + co) * 128 + ci] = __double2bfloat16((double)w[i] * sc);
  if (tap == 0 && ci == 0) {
    double b = cbias ? (double)cbias[co] : 0.0;
    if (gamma) b = (b - (double)mean[co]) * sc + (double)beta[co];
    bout[co] = (float)b;
  }
}

// stem: fp32 [128][4][3][3] -> bf16 [128][64], k = tap*4 + plane (rz_net_stem_tc's layout)
__global__ void rz_pack_stem_tc_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ ws) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 128 * 64) return;
  const int k = i & 63, co = i >> 6;
  float v = 0.0f;
  if (k < 36) { const int tap = k >> 2, pl = k & 3; v = w[((size_t)co * 4 + pl) * 9 + tap]; }
  ws[i] = __float2bfloat16_rn(v);
}
// Go stem: fp32 [128][17][3][3] -> bf16 [128][192], k = tap*17 + plane, zero from 153 (rz_net_stem_go_tc's layout)
__global__ void rz_pack_stem_go_tc_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ ws) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 128 * 192) return;
  const int k = i % 192, co = i / 192;
  float v = 0.0f;
  if (k < 153) { const int tap = k / 17, pl = k % 17; v = w[((size_t)co * 17 + pl) * 9 + tap]; }
  ws[i] = __float2bfloat16_rn(v);
}

// ---------------------------------------------------------------------------------------------------------
// row-parallel helpers: a warp owns a row (128 channels bf16 = 256 B), a lane 4 channels
// ---------------------------------------------------------------------------------------------------------
struct f4 { float v[4]; };
__device__ __forceinline__ f4 ld_bf16x4(const __nv_bfloat16* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  f4 r;
  r.v[0] = __uint_as_float(u.x << 16); r.v[1] = __uint_as_float(u.x & 0xffff0000u);
  r.v[2] = __uint_as_float(u.y << 16); r.v[3] = __uint_as_float(u.y & 0xffff0000u);
  return r;
}
__device__ __forceinline__ void st_bf16x4(__nv_bfloat16* p, const f4& r) {
  uint2 u;
  u.x = rz::pack_bf16x2(r.v[0], r.v[1]);
  u.y = rz::pack_bf16x2(r.v[2], r.v[3]);
  *reinterpret_cast<uint2*>(p) = u;
}
__device__ __forceinline__ bool row_on_board(long long row, int H, int W) {
  const int pos = (int)(row & 255);
  return (pos & 15) < W && (pos >> 4) < H;
}
// row r of the padded layout of stride kS (row = board*S*S + y*S + x) -> board, y, x
template <int kS>
__device__ __forceinline__ void row_pos(long long r, long long& b, int& y, int& x) {
  if (kS == 16) {
    const int pos = (int)(r & 255);
    b = r >> 8; y = pos >> 4; x = pos & 15;
  } else {
    b = r / (kS * kS);
    const int pos = (int)(r - b * (kS * kS));
    y = pos / kS; x = pos - y * kS;
  }
}
// a board square: x < W, y < H, and not one of the tail rows n*S*S .. round_up(n*S*S, 256) (there are none at S = 16)
template <int kS>
__device__ __forceinline__ bool row_on_board_s(long long r, int H, int W, long long n_valid) {
  long long b;
  int y, x;
  row_pos<kS>(r, b, y, x);
  return (kS == 16 || r < n_valid) && x < W && y < H;
}

// per-block partial sums of two per-channel quantities over the rows: part[blk][2][128]
//   kMode 0 (BatchNorm statistics):    s0 = sum y,    s1 = sum y^2
//   kMode 1 (BatchNorm backward):      s0 = sum dz,   s1 = sum dz * xhat,  dz = dout * (a > 0), xhat = (y - mean) * invstd
template <int kMode>
__global__ void __launch_bounds__(256)
rz_bn_reduce_kernel(const __nv_bfloat16* __restrict__ y, const __nv_bfloat16* __restrict__ dout,
                    const __nv_bfloat16* __restrict__ a, const float* __restrict__ mean,
                    const float* __restrict__ invstd, long long rows, float* __restrict__ part) {
  __shared__ float red[8][2][128];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, c0 = lane * 4;
  float s0[4] = {}, s1[4] = {};
  float mu[4] = {}, is[4] = {};
  if (kMode == 1) {
#pragma unroll
    for (int e = 0; e < 4; ++e) { mu[e] = mean[c0 + e]; is[e] = invstd[c0 + e]; }
  }
  for (long long r = (long long)blockIdx.x * 8 + warp; r < rows; r += (long long)gridDim.x * 8) {
    const f4 yv = ld_bf16x4(y + r * 128 + c0);
    if (kMode == 0) {
#pragma unroll
      for (int e = 0; e < 4; ++e) { s0[e] += yv.v[e]; s1[e] = fmaf(yv.v[e], yv.v[e], s1[e]); }
    } else {
      const f4 dv = ld_bf16x4(dout + r * 128 + c0), av = ld_bf16x4(a + r * 128 + c0);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float dz = av.v[e] > 0.0f ? dv.v[e] : 0.0f;
        s0[e] += dz;
        s1[e] = fmaf(dz, (yv.v[e] - mu[e]) * is[e], s1[e]);
      }
    }
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) { red[warp][0][c0 + e] = s0[e]; red[warp][1][c0 + e] = s1[e]; }
  __syncthreads();
  {
    const int which = threadIdx.x >> 7, c = threadIdx.x & 127;
    float t = 0.0f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w][which][c];
    part[((size_t)blockIdx.x * 2 + which) * 128 + c] = t;
  }
}

// fold the partials (in double) and produce the per-channel coefficients
//   mode 0: mean, invstd, scale = gamma * invstd, shift = beta - mean * scale; running statistics updated
//           (nn.BatchNorm2d in training mode: momentum 0.1, unbiased variance for running_var)
//   mode 1: dgamma, dbeta, c1 = dbeta / N, c2 = dgamma / N
//   mode 2: o0 = column sums
__global__ void __launch_bounds__(1024)
rz_bn_finalize_kernel(const float* __restrict__ part, int n_blocks, double count, int mode,
                      const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                      float momentum, float* __restrict__ running_mean, float* __restrict__ running_var,
                      float* __restrict__ o0, float* __restrict__ o1, float* __restrict__ o2,
                      float* __restrict__ o3) {
  // 8 slices of the partials are folded in parallel (fixed assignment and order: deterministic), then combined
  __shared__ double red[8][2][128];
  const int c = threadIdx.x & 127, sl = threadIdx.x >> 7;
  double s0 = 0.0, s1 = 0.0;
  for (int b = sl; b < n_blocks; b += 8) { s0 += part[((size_t)b * 2) * 128 + c]; s1 += part[((size_t)b * 2 + 1) * 128 + c]; }
  red[sl][0][c] = s0; red[sl][1][c] = s1;
  __syncthreads();
  if (sl != 0) return;
  s0 = 0.0; s1 = 0.0;
#pragma unroll
  for (int i = 0; i < 8; ++i) { s0 += red[i][0][c]; s1 += red[i][1][c]; }
  if (mode == 0) {
    const double mean = s0 / count;
    double var = s1 / count - mean * mean;
    if (var < 0.0) var = 0.0;
    const double invstd = 1.0 / sqrt(var + (double)eps);
    o0[c] = (float)mean; o1[c] = (float)invstd;
    const double sc = (double)gamma[c] * invstd;
    o2[c] = (float)sc; o3[c] = (float)((double)beta[c] - mean * sc);
    if (running_mean) {
      running_mean[c] = (1.0f - momentum) * running_mean[c] + momentum * (float)mean;
      running_var[c] = (1.0f - momentum) * running_var[c] + momentum * (float)(var * count / (count - 1.0));
    }
  } else if (mode == 1) {
    o0[c] = (float)s1;            // dgamma
    o1[c] = (float)s0;            // dbeta
    o2[c] = (float)(s0 / count);
    o3[c] = (float)(s1 / count);
  } else {
    o0[c] = (float)s0;            // plain column sums (a bias gradient)
  }
}

// a = relu(y * scale + shift (+ skip)), zero off the board
template <int kS>
__global__ void __launch_bounds__(256)
rz_bn_apply_kernel(const __nv_bfloat16* __restrict__ y, const float* __restrict__ scale, const float* __restrict__ shift,
                   const __nv_bfloat16* __restrict__ skip, __nv_bfloat16* __restrict__ out, long long rows,
                   long long n_valid, int H, int W) {
  const int lane = threadIdx.x & 31, c0 = lane * 4;
  float sc[4], sh[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) { sc[e] = scale[c0 + e]; sh[e] = shift[c0 + e]; }
  for (long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    f4 o;
    if (row_on_board_s<kS>(r, H, W, n_valid)) {
      const f4 yv = ld_bf16x4(y + r * 128 + c0);
#pragma unroll
      for (int e = 0; e < 4; ++e) o.v[e] = fmaf(yv.v[e], sc[e], sh[e]);
      if (skip) {
        const f4 sv = ld_bf16x4(skip + r * 128 + c0);
#pragma unroll
        for (int e = 0; e < 4; ++e) o.v[e] += sv.v[e];
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) o.v[e] = fmaxf(o.v[e], 0.0f);
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) o.v[e] = 0.0f;
    }
    st_bf16x4(out + r * 128 + c0, o);
  }
}

// dy = scale * (dz - c1 - xhat * c2), dz = dout * (a > 0); optionally dz itself (the gradient that flows into the skip)
template <int kS>
__global__ void __launch_bounds__(256)
rz_bn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ dout, const __nv_bfloat16* __restrict__ a,
                       const __nv_bfloat16* __restrict__ y, const float* __restrict__ mean,
                       const float* __restrict__ invstd, const float* __restrict__ scale, const float* __restrict__ c1,
                       const float* __restrict__ c2, __nv_bfloat16* __restrict__ dy, __nv_bfloat16* __restrict__ dz_out,
                       long long rows, long long n_valid, int H, int W) {
  const int lane = threadIdx.x & 31, c0 = lane * 4;
  float mu[4], is[4], sc[4], k1[4], k2[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) { mu[e] = mean[c0 + e]; is[e] = invstd[c0 + e]; sc[e] = scale[c0 + e]; k1[e] = c1[c0 + e]; k2[e] = c2[c0 + e]; }
  for (long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    f4 o, z;
    if (row_on_board_s<kS>(r, H, W, n_valid)) {
      const f4 dv = ld_bf16x4(dout + r * 128 + c0), av = ld_bf16x4(a + r * 128 + c0), yv = ld_bf16x4(y + r * 128 + c0);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        z.v[e] = av.v[e] > 0.0f ? dv.v[e] : 0.0f;
        o.v[e] = sc[e] * (z.v[e] - k1[e] - (yv.v[e] - mu[e]) * is[e] * k2[e]);
      }
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) { o.v[e] = 0.0f; z.v[e] = 0.0f; }
    }
    st_bf16x4(dy + r * 128 + c0, o);
    if (dz_out) st_bf16x4(dz_out + r * 128 + c0, z);
  }
}

// g = dout * (a > 0) (ReLU without BatchNorm: the stem)
__global__ void __launch_bounds__(256)
rz_relu_bwd_bf16_kernel(const __nv_bfloat16* __restrict__ dout, const __nv_bfloat16* __restrict__ a,
                        __nv_bfloat16* __restrict__ g, long long rows) {
  const int lane = threadIdx.x & 31, c0 = lane * 4;
  for (long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    const f4 dv = ld_bf16x4(dout + r * 128 + c0), av = ld_bf16x4(a + r * 128 + c0);
    f4 o;
#pragma unroll
    for (int e = 0; e < 4; ++e) o.v[e] = av.v[e] > 0.0f ? dv.v[e] : 0.0f;
    st_bf16x4(g + r * 128 + c0, o);
  }
}

// padded bf16 tile layout [round_up(n*S*S, 256)][128] <-> float32 [n][HW][128]
template <int kS>
__global__ void __launch_bounds__(256)
rz_tile_to_nhwc_kernel(const __nv_bfloat16* __restrict__ tile, float* __restrict__ out, int n, int H, int W) {
  const int lane = threadIdx.x & 31, c0 = lane * 4, HW = H * W;
  const long long rows = (long long)n * HW;
  for (long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    const int b = (int)(r / HW), pos = (int)(r - (long long)b * HW);
    const f4 v = ld_bf16x4(tile + ((long long)b * (kS * kS) + (pos / W) * kS + pos % W) * 128 + c0);
    *reinterpret_cast<float4*>(out + r * 128 + c0) = make_float4(v.v[0], v.v[1], v.v[2], v.v[3]);
  }
}
template <int kS>
__global__ void __launch_bounds__(256)
rz_nhwc_to_tile_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ tile, long long rows, int n, int H, int W) {
  const int lane = threadIdx.x & 31, c0 = lane * 4, HW = H * W;
  const long long n_valid = (long long)n * (kS * kS);
  for (long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    f4 o;
    if (row_on_board_s<kS>(r, H, W, n_valid)) {
      long long b;
      int y, x;
      row_pos<kS>(r, b, y, x);
      const float4 v = *reinterpret_cast<const float4*>(in + (b * HW + y * W + x) * 128 + c0);
      o.v[0] = v.x; o.v[1] = v.y; o.v[2] = v.z; o.v[3] = v.w;
    } else {
      o.v[0] = o.v[1] = o.v[2] = o.v[3] = 0.0f;
    }
    st_bf16x4(tile + r * 128 + c0, o);
  }
}

// float32 observation planes [n][n_planes][H][W] -> bf16 tile layout [round_up(n*S*S, 256)][128], channels
// 0..n_planes-1 (the rest zero): the stem's input as an operand of the tensor-core weight-gradient kernel (planes are
// 0/1: exact in bf16)
template <int kS>
__global__ void __launch_bounds__(256)
rz_planes_to_tile_kernel(const float* __restrict__ planes, int n_planes, __nv_bfloat16* __restrict__ tile, long long rows,
                         int n, int H, int W) {
  const int lane = threadIdx.x & 31, c0 = lane * 4, HW = H * W;
  const long long n_valid = (long long)n * (kS * kS);
  for (long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    f4 o;
    o.v[0] = o.v[1] = o.v[2] = o.v[3] = 0.0f;
    if (c0 < n_planes && row_on_board_s<kS>(r, H, W, n_valid)) {
      long long b;
      int y, x;
      row_pos<kS>(r, b, y, x);
      const float* src = planes + (b * n_planes + c0) * HW + y * W + x;
#pragma unroll
      for (int e = 0; e < 4; ++e) if (c0 + e < n_planes) o.v[e] = src[e * HW];
    }
    st_bf16x4(tile + r * 128 + c0, o);
  }
}

// float32 channels-last [n][HW][C] -> bf16 tiles carrying the value as a (high, low) pair, x = hi + lo to 16 mantissa
// bits: the operands of the float32-accurate weight gradient of the reference's own network on the tensor cores.
//   mode 0 (the layer input, 2C <= 128): tile_a[:, 0:C] = hi, tile_a[:, C:2C] = lo
//   mode 1 (the output gradient, C <= 128): tile_a[:, 0:C] = hi, tile_b[:, 0:C] = lo
__global__ void __launch_bounds__(256)
rz_nhwc_to_tile_hilo_kernel(const float* __restrict__ in, int C_total, int c_off, int C, __nv_bfloat16* __restrict__ tile_a,
                            __nv_bfloat16* __restrict__ tile_b, int mode, int n, int H, int W) {
  const int lane = threadIdx.x & 31, c0 = lane * 4, HW = H * W;
  const long long rows = (long long)n * 256;
  for (long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    f4 a, b;
#pragma unroll
    for (int e = 0; e < 4; ++e) { a.v[e] = 0.0f; b.v[e] = 0.0f; }
    if (row_on_board(r, H, W)) {
      const int pos = (int)(r & 255);
      const float* src = in + ((r >> 8) * HW + (pos >> 4) * W + (pos & 15)) * C_total + c_off;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int c = c0 + e;
        const int cs = c < C ? c : c - C;
        if (c < C || (mode == 0 && c < 2 * C)) {
          const float x = src[cs];
          const float hi = __bfloat162float(__float2bfloat16_rn(x));
          if (c < C) { a.v[e] = hi; b.v[e] = x - hi; }
          else a.v[e] = x - hi;
        }
      }
    }
    st_bf16x4(tile_a + r * 128 + c0, a);
    if (mode == 1) st_bf16x4(tile_b + r * 128 + c0, b);
  }
}

// float32 tile [n*256][128] (first C channels) -> float32 channels-last [n][HW][C]
__global__ void __launch_bounds__(256)
rz_tile_f32_to_nhwc_kernel(const float* __restrict__ tile, float* __restrict__ out, int C, int n, int H, int W) {
  const int lane = threadIdx.x & 31, HW = H * W;
  const long long rows = (long long)n * HW;
  for (long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    const int b = (int)(r / HW), pos = (int)(r - (long long)b * HW);
    const float* src = tile + ((long long)b * 256 + (pos / W) * 16 + pos % W) * 128;
    for (int c = lane; c < C; c += 32) out[r * C + c] = src[c];
  }
}

// the data gradient of a float32-accurate layer back in tile space: g = (grad_a + grad_b) * (act > 0) on the first C
// channels (act: the layer's activation as a [hi | lo ...] pair tile, its sign is the sign of the high part); g is
// written back to grad_a as float32 (for the bias gradient) and as bf16 pairs: pair_out = [hi | lo] in one tile (the
// input of the next data gradient; may be NULL), hi_out / lo_out = the two gradient tiles of the weight gradient
__global__ void __launch_bounds__(256)
rz_tile_grad_mask_split_kernel(float* __restrict__ grad_a, const float* __restrict__ grad_b,
                               const __nv_bfloat16* __restrict__ act, int C, __nv_bfloat16* __restrict__ pair_out,
                               __nv_bfloat16* __restrict__ hi_out, __nv_bfloat16* __restrict__ lo_out, long long rows) {
  const int lane = threadIdx.x & 31, c0 = lane * 4;
  for (long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    f4 hi, lo, pr;
    float g[4];
    const f4 av = ld_bf16x4(act + r * 128 + (c0 < C ? c0 : 0));
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int c = c0 + e;
      g[e] = 0.0f;
      if (c < C) {
        float x = grad_a[r * 128 + c] + (grad_b ? grad_b[r * 128 + c] : 0.0f);
        g[e] = av.v[e] > 0.0f ? x : 0.0f;
      }
      hi.v[e] = __bfloat162float(__float2bfloat16_rn(g[e]));
      lo.v[e] = g[e] - hi.v[e];
    }
    if (c0 < C) {
#pragma unroll
      for (int e = 0; e < 4; ++e) if (c0 + e < C) grad_a[r * 128 + c0 + e] = g[e];
    }
    st_bf16x4(hi_out + r * 128 + c0, hi);
    st_bf16x4(lo_out + r * 128 + c0, lo);
    if (pair_out) {
      // channel c of the pair tile: hi for c < C, lo of channel c - C for C <= c < 2C (C is a multiple of 4): the low
      // parts come from the lane that owns those channels
      const int src_lane = lane - (C >> 2);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float lo_other = __shfl_sync(RZ_FULL, lo.v[e], src_lane < 0 ? 0 : src_lane);
        pr.v[e] = c0 < C ? hi.v[e] : (c0 < 2 * C ? lo_other : 0.0f);
      }
      st_bf16x4(pair_out + r * 128 + c0, pr);
    }
  }
}

inline int row_grid(long long rows) {
  long long b = (rows + 7) / 8;
  return (int)(b < 1 ? 1 : (b > 148 * 8 ? 148 * 8 : b));
}
constexpr int BN_BLOCKS = 148 * 2;

// rows of a tensor in the padded layout of stride S: round_up(n*S*S, 256) (n*256 at S = 16)
inline long long layout_rows(int n_boards, int S) { return ((long long)n_boards * S * S + 255) / 256 * 256; }

template <int kS>
int wgrad_launch(const void* x, const void* dy, float* dw_oihw, float* scratch, int n_boards, int splits, int n_tiles,
                 cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(rz_conv_wgrad_tc_kernel<kS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         WgGeo<kS>::SMEM);
    if (e != cudaSuccess) { rz_set_error("rz_learn_conv_wgrad_tc_ex: smem attribute: %s", cudaGetErrorString(e)); return -2; }
    attr_set = true;
  }
  // the tensor maps end at n*S*S rows: TMA fills the halo before row 0 and a partial last tile with zeros
  CUtensorMap tmap_x, tmap_dy;
  if (rz::make_tmap_2d(&tmap_x, x, (uint64_t)n_boards * kS * kS, 128, WgGeo<kS>::XROWS)) return -1;
  if (rz::make_tmap_2d(&tmap_dy, dy, (uint64_t)n_boards * kS * kS, 128, WG_TILE)) return -1;
  WgradParams p;
  p.part = scratch; p.n_tiles = n_tiles; p.n_splits = splits;
  rz_conv_wgrad_tc_kernel<kS><<<splits * 3, WG_THREADS, WgGeo<kS>::SMEM, st>>>(tmap_x, tmap_dy, p);
  rz_wgrad_tc_final_kernel<<<(9 * 128 * 128 + 255) / 256, 256, 0, st>>>(scratch, dw_oihw, splits);
  RZ_LAUNCH_CHECK("rz_learn_conv_wgrad_tc_ex");
  return 0;
}

}  // namespace

#define RZ_REQUIRE_STRIDE(fn, S) RZ_REQUIRE((S) == 16 || (S) == 20, fn ": row_stride %d (16 or 20)", (S))
#define RZ_REQUIRE_BOARD(fn, H, W, S)                                                                              \
  RZ_REQUIRE((H) >= 1 && (H) < (S) && (W) >= 1 && (W) < (S), fn ": board %dx%d does not fit row_stride %d", (H), (W), (S))

// =========================================================================================================
// C ABI
// =========================================================================================================
extern "C" int rz_learn_conv_wgrad_tc_ex(const void* x, const void* dy, float* dw_oihw, float* scratch,
                                         long long scratch_floats, int n_boards, int row_stride, int n_ctas,
                                         void* stream) {
  RZ_REQUIRE(x && dy && dw_oihw && scratch && n_boards >= 1, "rz_learn_conv_wgrad_tc_ex: bad arguments");
  RZ_REQUIRE_STRIDE("rz_learn_conv_wgrad_tc_ex", row_stride);
  int ctas = n_ctas > 0 ? n_ctas : 147;
  ctas = ctas / 3 * 3;
  if (ctas < 3) ctas = 3;
  const long long n_tiles = ((long long)n_boards * row_stride * row_stride + WG_TILE - 1) / WG_TILE;
  RZ_REQUIRE(n_tiles < (1LL << 30), "rz_learn_conv_wgrad_tc_ex: %d boards", n_boards);
  int splits = ctas / 3;
  if (splits > n_tiles) splits = (int)n_tiles;
  RZ_REQUIRE(scratch_floats >= (long long)splits * 9 * 128 * 128, "rz_learn_conv_wgrad_tc_ex: scratch holds %lld floats, %lld needed",
             scratch_floats, (long long)splits * 9 * 128 * 128);
  cudaStream_t st = (cudaStream_t)stream;
  return row_stride == 16 ? wgrad_launch<16>(x, dy, dw_oihw, scratch, n_boards, splits, (int)n_tiles, st)
                          : wgrad_launch<20>(x, dy, dw_oihw, scratch, n_boards, splits, (int)n_tiles, st);
}

extern "C" int rz_learn_conv_wgrad_tc(const void* x, const void* dy, float* dw_oihw, float* scratch,
                                      long long scratch_floats, int n_boards, int n_ctas, void* stream) {
  return rz_learn_conv_wgrad_tc_ex(x, dy, dw_oihw, scratch, scratch_floats, n_boards, 16, n_ctas, stream);
}

extern "C" int rz_learn_pack_conv_tc(const float* w_oihw, void* w_fwd, void* w_bwd, void* stream) {
  RZ_REQUIRE(w_oihw && w_fwd && w_bwd, "rz_learn_pack_conv_tc: null argument");
  rz_pack_conv_tc_kernel<<<(128 * 128 * 9 + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
      w_oihw, (__nv_bfloat16*)w_fwd, (__nv_bfloat16*)w_bwd);
  RZ_LAUNCH_CHECK("rz_learn_pack_conv_tc");
  return 0;
}

extern "C" int rz_net_pack_conv_bn_tc(const float* w_oihw, const float* conv_bias, const float* gamma, const float* beta,
                                      const float* running_mean, const float* running_var, float eps, void* w_out,
                                      float* b_out, void* stream) {
  RZ_REQUIRE(w_oihw && w_out && b_out, "rz_net_pack_conv_bn_tc: null argument");
  RZ_REQUIRE(!gamma || (beta && running_mean && running_var), "rz_net_pack_conv_bn_tc: incomplete BatchNorm");
  rz_pack_conv_bn_tc_kernel<<<(128 * 128 * 9 + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
      w_oihw, conv_bias, gamma, beta, running_mean, running_var, eps, (__nv_bfloat16*)w_out, b_out);
  RZ_LAUNCH_CHECK("rz_net_pack_conv_bn_tc");
  return 0;
}

extern "C" int rz_learn_pack_stem_tc_ex(const float* w_oihw, int in_planes, void* w_stem, void* stream) {
  RZ_REQUIRE(w_oihw && w_stem, "rz_learn_pack_stem_tc_ex: null argument");
  RZ_REQUIRE(in_planes == 4 || in_planes == 17, "rz_learn_pack_stem_tc_ex: in_planes %d (4 or 17)", in_planes);
  if (in_planes == 4)
    rz_pack_stem_tc_kernel<<<(128 * 64 + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w_oihw, (__nv_bfloat16*)w_stem);
  else
    rz_pack_stem_go_tc_kernel<<<(128 * 192 + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w_oihw, (__nv_bfloat16*)w_stem);
  RZ_LAUNCH_CHECK("rz_learn_pack_stem_tc_ex");
  return 0;
}

extern "C" int rz_learn_pack_stem_tc(const float* w_oihw, void* w_stem, void* stream) {
  return rz_learn_pack_stem_tc_ex(w_oihw, 4, w_stem, stream);
}

extern "C" int rz_learn_bn_forward_ex(const void* y, const void* skip, void* out, const float* gamma, const float* beta,
                                      float* running_mean, float* running_var, float eps, float momentum, float* stats,
                                      float* scratch, int n_boards, int board_rows, int board_cols, int row_stride,
                                      void* stream) {
  RZ_REQUIRE(y && out && gamma && beta && stats && scratch && n_boards >= 1, "rz_learn_bn_forward_ex: bad arguments");
  RZ_REQUIRE_STRIDE("rz_learn_bn_forward_ex", row_stride);
  RZ_REQUIRE_BOARD("rz_learn_bn_forward_ex", board_rows, board_cols, row_stride);
  const long long rows = layout_rows(n_boards, row_stride), n_valid = (long long)n_boards * row_stride * row_stride;
  const int blocks = row_grid(rows) < BN_BLOCKS ? row_grid(rows) : BN_BLOCKS;
  cudaStream_t st = (cudaStream_t)stream;
  rz_bn_reduce_kernel<0><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)y, nullptr, nullptr, nullptr, nullptr, rows, scratch);
  // stats: [4][128] = mean, invstd, scale, shift
  rz_bn_finalize_kernel<<<1, 1024, 0, st>>>(scratch, blocks, (double)n_boards * board_rows * board_cols, 0, gamma, beta, eps,
                                          momentum, running_mean, running_var, stats, stats + 128, stats + 256, stats + 384);
  if (row_stride == 16)
    rz_bn_apply_kernel<16><<<row_grid(rows), 256, 0, st>>>((const __nv_bfloat16*)y, stats + 256, stats + 384,
                                                          (const __nv_bfloat16*)skip, (__nv_bfloat16*)out, rows, n_valid,
                                                          board_rows, board_cols);
  else
    rz_bn_apply_kernel<20><<<row_grid(rows), 256, 0, st>>>((const __nv_bfloat16*)y, stats + 256, stats + 384,
                                                          (const __nv_bfloat16*)skip, (__nv_bfloat16*)out, rows, n_valid,
                                                          board_rows, board_cols);
  RZ_LAUNCH_CHECK("rz_learn_bn_forward_ex");
  return 0;
}

extern "C" int rz_learn_bn_forward(const void* y, const void* skip, void* out, const float* gamma, const float* beta,
                                   float* running_mean, float* running_var, float eps, float momentum, float* stats,
                                   float* scratch, int n_boards, int board_rows, int board_cols, void* stream) {
  return rz_learn_bn_forward_ex(y, skip, out, gamma, beta, running_mean, running_var, eps, momentum, stats, scratch,
                                n_boards, board_rows, board_cols, 16, stream);
}

extern "C" int rz_learn_bn_backward_ex(const void* dout, const void* act, const void* y, const float* stats, float* dgamma,
                                       float* dbeta, void* dy, void* dz_out, float* scratch, int n_boards, int board_rows,
                                       int board_cols, int row_stride, void* stream) {
  RZ_REQUIRE(dout && act && y && stats && dgamma && dbeta && dy && scratch && n_boards >= 1, "rz_learn_bn_backward_ex: bad arguments");
  RZ_REQUIRE_STRIDE("rz_learn_bn_backward_ex", row_stride);
  RZ_REQUIRE_BOARD("rz_learn_bn_backward_ex", board_rows, board_cols, row_stride);
  const long long rows = layout_rows(n_boards, row_stride), n_valid = (long long)n_boards * row_stride * row_stride;
  const int blocks = row_grid(rows) < BN_BLOCKS ? row_grid(rows) : BN_BLOCKS;
  cudaStream_t st = (cudaStream_t)stream;
  rz_bn_reduce_kernel<1><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)y, (const __nv_bfloat16*)dout, (const __nv_bfloat16*)act,
                                                stats, stats + 128, rows, scratch);
  float* coef = scratch + (size_t)BN_BLOCKS * 256;        // c1, c2
  rz_bn_finalize_kernel<<<1, 1024, 0, st>>>(scratch, blocks, (double)n_boards * board_rows * board_cols, 1, nullptr, nullptr, 0.0f,
                                          0.0f, nullptr, nullptr, dgamma, dbeta, coef, coef + 128);
  if (row_stride == 16)
    rz_bn_bwd_apply_kernel<16><<<row_grid(rows), 256, 0, st>>>((const __nv_bfloat16*)dout, (const __nv_bfloat16*)act,
                                                              (const __nv_bfloat16*)y, stats, stats + 128, stats + 256, coef,
                                                              coef + 128, (__nv_bfloat16*)dy, (__nv_bfloat16*)dz_out, rows,
                                                              n_valid, board_rows, board_cols);
  else
    rz_bn_bwd_apply_kernel<20><<<row_grid(rows), 256, 0, st>>>((const __nv_bfloat16*)dout, (const __nv_bfloat16*)act,
                                                              (const __nv_bfloat16*)y, stats, stats + 128, stats + 256, coef,
                                                              coef + 128, (__nv_bfloat16*)dy, (__nv_bfloat16*)dz_out, rows,
                                                              n_valid, board_rows, board_cols);
  RZ_LAUNCH_CHECK("rz_learn_bn_backward_ex");
  return 0;
}

extern "C" int rz_learn_bn_backward(const void* dout, const void* act, const void* y, const float* stats, float* dgamma,
                                    float* dbeta, void* dy, void* dz_out, float* scratch, int n_boards, int board_rows,
                                    int board_cols, void* stream) {
  return rz_learn_bn_backward_ex(dout, act, y, stats, dgamma, dbeta, dy, dz_out, scratch, n_boards, board_rows, board_cols,
                                 16, stream);
}

extern "C" int rz_learn_planes_to_tile_ex(const float* planes, int n_planes, void* tile, int n_boards, int board_rows,
                                          int board_cols, int row_stride, void* stream) {
  RZ_REQUIRE(planes && tile && n_boards >= 1, "rz_learn_planes_to_tile_ex: bad arguments");
  RZ_REQUIRE(n_planes == 4 || n_planes == 17, "rz_learn_planes_to_tile_ex: n_planes %d (4 or 17)", n_planes);
  RZ_REQUIRE_STRIDE("rz_learn_planes_to_tile_ex", row_stride);
  RZ_REQUIRE_BOARD("rz_learn_planes_to_tile_ex", board_rows, board_cols, row_stride);
  const long long rows = layout_rows(n_boards, row_stride);
  cudaStream_t st = (cudaStream_t)stream;
  if (row_stride == 16)
    rz_planes_to_tile_kernel<16><<<row_grid(rows), 256, 0, st>>>(planes, n_planes, (__nv_bfloat16*)tile, rows, n_boards,
                                                                board_rows, board_cols);
  else
    rz_planes_to_tile_kernel<20><<<row_grid(rows), 256, 0, st>>>(planes, n_planes, (__nv_bfloat16*)tile, rows, n_boards,
                                                                board_rows, board_cols);
  RZ_LAUNCH_CHECK("rz_learn_planes_to_tile_ex");
  return 0;
}

extern "C" int rz_learn_planes_to_tile(const float* planes, void* tile, int n_boards, int board_rows, int board_cols,
                                       void* stream) {
  return rz_learn_planes_to_tile_ex(planes, 4, tile, n_boards, board_rows, board_cols, 16, stream);
}

extern "C" int rz_learn_nhwc_to_tile_hilo(const float* in, int channels, void* tile_a, void* tile_b, int mode, int n_boards,
                                          int board_rows, int board_cols, void* stream) {
  RZ_REQUIRE(in && tile_a && (mode == 0 || tile_b) && n_boards >= 1 && board_rows <= 15 && board_cols <= 15,
             "rz_learn_nhwc_to_tile_hilo: bad arguments");
  RZ_REQUIRE((mode == 0 && channels >= 1 && 2 * channels <= 128) || (mode == 1 && channels >= 1 && channels <= 128),
             "rz_learn_nhwc_to_tile_hilo: mode %d with %d channels", mode, channels);
  rz_nhwc_to_tile_hilo_kernel<<<row_grid((long long)n_boards * 256), 256, 0, (cudaStream_t)stream>>>(
      in, channels, 0, channels, (__nv_bfloat16*)tile_a, (__nv_bfloat16*)tile_b, mode, n_boards, board_rows, board_cols);
  RZ_LAUNCH_CHECK("rz_learn_nhwc_to_tile_hilo");
  return 0;
}

extern "C" int rz_learn_nhwc_to_tile_hilo_slice(const float* in, int channels_total, int channel_offset, int channels,
                                                void* tile_a, int n_boards, int board_rows, int board_cols, void* stream) {
  RZ_REQUIRE(in && tile_a && n_boards >= 1 && board_rows <= 15 && board_cols <= 15 && channels >= 1 && 2 * channels <= 128 &&
             channel_offset >= 0 && channel_offset + channels <= channels_total, "rz_learn_nhwc_to_tile_hilo_slice: bad arguments");
  rz_nhwc_to_tile_hilo_kernel<<<row_grid((long long)n_boards * 256), 256, 0, (cudaStream_t)stream>>>(
      in, channels_total, channel_offset, channels, (__nv_bfloat16*)tile_a, nullptr, 0, n_boards, board_rows, board_cols);
  RZ_LAUNCH_CHECK("rz_learn_nhwc_to_tile_hilo_slice");
  return 0;
}

extern "C" int rz_learn_tile_f32_to_nhwc(const float* tile, float* out, int channels, int n_boards, int board_rows,
                                         int board_cols, void* stream) {
  RZ_REQUIRE(tile && out && n_boards >= 1 && board_rows <= 15 && board_cols <= 15 && channels >= 1 && channels <= 128,
             "rz_learn_tile_f32_to_nhwc: bad arguments");
  rz_tile_f32_to_nhwc_kernel<<<row_grid((long long)n_boards * board_rows * board_cols), 256, 0, (cudaStream_t)stream>>>(
      tile, out, channels, n_boards, board_rows, board_cols);
  RZ_LAUNCH_CHECK("rz_learn_tile_f32_to_nhwc");
  return 0;
}

extern "C" int rz_learn_tile_grad_mask_split(float* grad_a, const float* grad_b, const void* act_pair, int channels,
                                             void* pair_out, void* hi_out, void* lo_out, int n_boards, void* stream) {
  RZ_REQUIRE(grad_a && act_pair && hi_out && lo_out && n_boards >= 1 && channels >= 1 && 2 * channels <= 128,
             "rz_learn_tile_grad_mask_split: bad arguments");
  rz_tile_grad_mask_split_kernel<<<row_grid((long long)n_boards * 256), 256, 0, (cudaStream_t)stream>>>(
      grad_a, grad_b, (const __nv_bfloat16*)act_pair, channels, (__nv_bfloat16*)pair_out, (__nv_bfloat16*)hi_out,
      (__nv_bfloat16*)lo_out, (long long)n_boards * 256);
  RZ_LAUNCH_CHECK("rz_learn_tile_grad_mask_split");
  return 0;
}

extern "C" int rz_learn_tile_colsum_ex(const void* tile, float* out, float* scratch, int n_boards, int row_stride,
                                       void* stream) {
  RZ_REQUIRE(tile && out && scratch && n_boards >= 1, "rz_learn_tile_colsum_ex: bad arguments");
  RZ_REQUIRE_STRIDE("rz_learn_tile_colsum_ex", row_stride);
  const long long rows = layout_rows(n_boards, row_stride);
  const int blocks = row_grid(rows) < BN_BLOCKS ? row_grid(rows) : BN_BLOCKS;
  cudaStream_t st = (cudaStream_t)stream;
  rz_bn_reduce_kernel<0><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)tile, nullptr, nullptr, nullptr, nullptr, rows, scratch);
  rz_bn_finalize_kernel<<<1, 1024, 0, st>>>(scratch, blocks, 1.0, 2, nullptr, nullptr, 0.0f, 0.0f, nullptr, nullptr, out, nullptr,
                                           nullptr, nullptr);
  RZ_LAUNCH_CHECK("rz_learn_tile_colsum_ex");
  return 0;
}

extern "C" int rz_learn_tile_colsum(const void* tile, float* out, float* scratch, int n_boards, void* stream) {
  return rz_learn_tile_colsum_ex(tile, out, scratch, n_boards, 16, stream);
}

extern "C" int rz_learn_relu_bwd_bf16_ex(const void* dout, const void* act, void* grad, int n_boards, int row_stride,
                                         void* stream) {
  RZ_REQUIRE(dout && act && grad && n_boards >= 1, "rz_learn_relu_bwd_bf16_ex: bad arguments");
  RZ_REQUIRE_STRIDE("rz_learn_relu_bwd_bf16_ex", row_stride);
  const long long rows = layout_rows(n_boards, row_stride);
  rz_relu_bwd_bf16_kernel<<<row_grid(rows), 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)dout, (const __nv_bfloat16*)act,
                                                                            (__nv_bfloat16*)grad, rows);
  RZ_LAUNCH_CHECK("rz_learn_relu_bwd_bf16_ex");
  return 0;
}

extern "C" int rz_learn_relu_bwd_bf16(const void* dout, const void* act, void* grad, int n_boards, void* stream) {
  return rz_learn_relu_bwd_bf16_ex(dout, act, grad, n_boards, 16, stream);
}

extern "C" int rz_learn_tile_to_nhwc_ex(const void* tile, float* out, int n_boards, int board_rows, int board_cols,
                                        int row_stride, void* stream) {
  RZ_REQUIRE(tile && out && n_boards >= 1, "rz_learn_tile_to_nhwc_ex: bad arguments");
  RZ_REQUIRE_STRIDE("rz_learn_tile_to_nhwc_ex", row_stride);
  RZ_REQUIRE_BOARD("rz_learn_tile_to_nhwc_ex", board_rows, board_cols, row_stride);
  const int grid = row_grid((long long)n_boards * board_rows * board_cols);
  cudaStream_t st = (cudaStream_t)stream;
  if (row_stride == 16)
    rz_tile_to_nhwc_kernel<16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)tile, out, n_boards, board_rows, board_cols);
  else
    rz_tile_to_nhwc_kernel<20><<<grid, 256, 0, st>>>((const __nv_bfloat16*)tile, out, n_boards, board_rows, board_cols);
  RZ_LAUNCH_CHECK("rz_learn_tile_to_nhwc_ex");
  return 0;
}

extern "C" int rz_learn_tile_to_nhwc(const void* tile, float* out, int n_boards, int board_rows, int board_cols, void* stream) {
  return rz_learn_tile_to_nhwc_ex(tile, out, n_boards, board_rows, board_cols, 16, stream);
}

extern "C" int rz_learn_nhwc_to_tile_ex(const float* in, void* tile, int n_boards, int board_rows, int board_cols,
                                        int row_stride, void* stream) {
  RZ_REQUIRE(in && tile && n_boards >= 1, "rz_learn_nhwc_to_tile_ex: bad arguments");
  RZ_REQUIRE_STRIDE("rz_learn_nhwc_to_tile_ex", row_stride);
  RZ_REQUIRE_BOARD("rz_learn_nhwc_to_tile_ex", board_rows, board_cols, row_stride);
  const long long rows = layout_rows(n_boards, row_stride);
  cudaStream_t st = (cudaStream_t)stream;
  if (row_stride == 16)
    rz_nhwc_to_tile_kernel<16><<<row_grid(rows), 256, 0, st>>>(in, (__nv_bfloat16*)tile, rows, n_boards, board_rows, board_cols);
  else
    rz_nhwc_to_tile_kernel<20><<<row_grid(rows), 256, 0, st>>>(in, (__nv_bfloat16*)tile, rows, n_boards, board_rows, board_cols);
  RZ_LAUNCH_CHECK("rz_learn_nhwc_to_tile_ex");
  return 0;
}

extern "C" int rz_learn_nhwc_to_tile(const float* in, void* tile, int n_boards, int board_rows, int board_cols, void* stream) {
  return rz_learn_nhwc_to_tile_ex(in, tile, n_boards, board_rows, board_cols, 16, stream);
}
